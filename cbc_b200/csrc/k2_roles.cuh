/*
 * k2_roles.cuh -- K2 for blocked containers (format v4): one SCALAR coder per (block, substream).
 *
 * Replaces, bit for bit per substream (include/cbcg_format.h, "Substreams of a block"):
 *   stream_model.c       update_model :31-51, send_value_to_as :53-76, read_value_from_as :78-117
 *   Arithmetic_stream.c  arithmetic_encoder_step :274-345, arithmetic_get_symbol_range :373-381,
 *                        arithmetic_decoder_step :389-454, the MSB-first bit packer :155-194
 *   read_compression.c   compress_read :15-44, compress_pos(_alpha) :75-159, compress_flag :50-70,
 *                        compress_match/snps/indels/var/chars :164-260, the emission half of compress_edits :557-600,
 *                        compute_delta_to_first_snp :703-718
 *   read_decompression.c decompress_read :59-86 and the decoding half of reconstruct_read :339-458
 *
 * A block's symbols are split by model group into four independent arithmetic-coded substreams (POS | FLAG |
 * match + counts | var + bases), and each (block, substream) is coded here by one scalar coder. Encode: the four are
 * independent. Decode runs {POS, FLAG} -> {match, counts} -> {var, bases}: the match context needs samePos, the edit
 * loops need the counts, and the base context needs the reference base under the decoded position. Models live where
 * the merge kernels expect them (the block's WarpModels image, its workspace: k2_layout.h).
 *
 * Everything here is plain scalar C++ marked host + device. It is the reference the GPU's substream kernels are held
 * to: tests/native/test_k2_roles.cpp runs it on the CPU against the oracle's containers (the warp-cooperative kernels
 * can only be checked on a GPU). On the device, the interval kernel of a two-kernel encode (k2_blocks.cu) codes with
 * K2Ac, and k2_snapshot_init writes the initial generation snapshot.
 */
#pragma once
#include <string.h>
#include "k2_layout.h"
#include "ac_core.h"
#include "internal.h"

#define K2R_LIKELY(c)   __builtin_expect(!!(c), 1)
#define K2R_UNLIKELY(c) __builtin_expect(!!(c), 0)

struct K2U4 { uint32_t x, y, z, w; };
/* four counts of a 16-byte aligned row */
K2_HD K2U4 k2_ld4(const uint32_t *p) {
#ifdef __CUDA_ARCH__
    const uint4 v = *reinterpret_cast<const uint4 *>(p);
    K2U4 r = { v.x, v.y, v.z, v.w };
    return r;
#else
    K2U4 r = { p[0], p[1], p[2], p[3] };
    return r;
#endif
}
K2_HD void k2_add_u32(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicAdd(p, v);
#else
    *p += v;
#endif
}
K2_HD uint32_t k2_base_code(uint32_t c) { return c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u; }

/* ------------------------------------------------------------------------------------------------ arithmetic coder */
struct K2Ac {
    AcInterval a; uint32_t t; int32_t scale3;
    uint64_t acc; uint32_t nacc, out_pos, out_cap; uint8_t *out;            /* encoder: MSB-first packer, 32 bits at a time */
    const uint8_t *in; uint32_t in_pos, in_len, dcnt; uint64_t dbuf;        /* decoder: upcoming bits, left-aligned */
    int err; uint32_t nsym;

    K2_HD void init_enc(uint8_t *o, uint32_t cap) {
        a.l = 0; a.u = CBCG_AC_TOP; t = 0; scale3 = 0; acc = 0; nacc = 0; out_pos = 0; out_cap = cap; out = o;
        in = nullptr; in_pos = in_len = dcnt = 0; dbuf = 0; err = 0; nsym = 0;
    }
    K2_HD void init_dec(const uint8_t *i, uint32_t len) {
        a.l = 0; a.u = CBCG_AC_TOP; scale3 = 0; acc = 0; nacc = 0; out_pos = 0; out_cap = 0; out = nullptr;
        in = i; in_pos = 0; in_len = len; dcnt = 0; dbuf = 0; err = 0; nsym = 0;
        t = get_bits(CBCG_AC_BITS);                                          /* src/Arithmetic_stream.c:262 */
    }
    K2_HD void put_bits(uint32_t v, uint32_t k) {                            /* k <= 32 */
        if (k == 0) return;
        acc = (acc << k) | (uint64_t)v;
        nacc += k;
        if (nacc >= 32u) {
            const uint32_t w = (uint32_t)(acc >> (nacc - 32u));
            if (out_pos + 4u <= out_cap) {
#ifdef __CUDA_ARCH__
                *reinterpret_cast<uint32_t *>(out + out_pos) = __byte_perm(w, 0u, 0x0123);   /* the region is 16-byte aligned */
#else
                out[out_pos] = (uint8_t)(w >> 24); out[out_pos + 1] = (uint8_t)(w >> 16); out[out_pos + 2] = (uint8_t)(w >> 8); out[out_pos + 3] = (uint8_t)w;
#endif
            } else err = CBCG_ERR_CAPACITY;
            out_pos += 4u;
            nacc -= 32u;
            acc &= (1ull << nacc) - 1ull;
        }
    }
    /* one bit b0, `run` copies of its inverse (the pending E3 bits, :318-322), then the low rest_bits of rest */
    K2_HD void emit(uint32_t b0, uint32_t run, uint32_t rest, uint32_t rest_bits) {
        if (K2R_LIKELY(run + 1u + rest_bits <= 32u)) {
            const uint32_t inv = b0 ? 0u : 0xffffffffu;
            put_bits((b0 << (run + rest_bits)) | ((inv & ((1u << run) - 1u)) << rest_bits) | rest, run + 1u + rest_bits);
            return;
        }
        const uint32_t inv = b0 ? 0u : 0xffffffffu;
        uint32_t r = run < 31u ? run : 31u;
        put_bits((b0 << r) | (inv & ((1u << r) - 1u)), r + 1u);
        run -= r;
        while (run) { r = run < 32u ? run : 32u; put_bits(r == 32u ? inv : (inv & ((1u << r) - 1u)), r); run -= r; }
        put_bits(rest, rest_bits);
    }
    K2_HD uint32_t get_bits(uint32_t k) {                                    /* k <= 32; zeros past the end */
        if (k == 0) return 0u;
        if (dcnt < k) {
            uint32_t w = 0;
            for (uint32_t i = 0; i < 4u; i++) { w <<= 8; if (in_pos + i < in_len) w |= (uint32_t)in[in_pos + i]; }
            in_pos += 4u;
            dbuf |= (uint64_t)w << (32u - dcnt);
            dcnt += 32u;
        }
        const uint32_t r = (uint32_t)(dbuf >> (64u - k));
        dbuf <<= k;
        dcnt -= k;
        return r;
    }
    K2_HD void encode(uint32_t lo, uint32_t cnt, uint32_t n) {
        if (K2R_UNLIKELY(cnt == 0u || n == 0u)) { err = CBCG_ERR_INPUT; return; }      /* reference: assert :71 / :293 */
        ac_narrow(a, lo, lo + cnt, n);
        uint32_t k, bits, m; AcInterval nx;
        ac_renorm_shape(a, k, bits, m, nx);
        if (k) { emit((bits >> (k - 1u)) & 1u, (uint32_t)scale3, bits & ((1u << (k - 1u)) - 1u), k - 1u); scale3 = 0; }
        scale3 += (int32_t)m;
        a = nx;
        nsym++;
    }
    K2_HD void decode_step(uint32_t lo, uint32_t cnt, uint32_t n) {
        ac_narrow(a, lo, lo + cnt, n);
        uint32_t k, bits, m; AcInterval nx;
        ac_renorm_shape(a, k, bits, m, nx);
        uint32_t s = k + m;                                                   /* up to 51 bits; the tag keeps the last 26 */
        uint64_t in64 = 0;
        while (s) { const uint32_t take = s < 32u ? s : 32u; in64 = (in64 << take) | get_bits(take); s -= take; }
        t = ac_tag_shift(t, k, m, (uint32_t)in64);
        a = nx;
        nsym++;
    }
    /* 1 + pending bits, zeros ever after (the decoder reads zeros past the end); nothing coded: nothing stored */
    K2_HD uint32_t finish_short() {
        if (nsym == 0) return 0u;
        emit(1u, (uint32_t)scale3, 0u, 0u);
        scale3 = 0;
        const uint32_t full = nacc >> 3, rem = nacc & 7u;
        for (uint32_t i = 0; i < full; i++) {
            const uint32_t byte = (uint32_t)(acc >> (nacc - 8u * (i + 1u))) & 0xffu;
            if (out_pos < out_cap) out[out_pos] = (uint8_t)byte; else err = CBCG_ERR_CAPACITY;
            out_pos++;
        }
        if (rem) {
            const uint32_t last = ((uint32_t)acc & ((1u << rem) - 1u)) << (8u - rem);
            if (out_pos < out_cap) out[out_pos] = (uint8_t)last; else err = CBCG_ERR_CAPACITY;
            out_pos++;
        }
        nacc = 0; acc = 0;
        return out_pos;
    }
    /* decoder search without the division of arithmetic_get_symbol_range (:373-381): for a cumulative count c,
       c <= target  <=>  c * range <= A  with  A = (t - l + 1) n - 1 */
    K2_HD uint64_t dec_A(uint32_t n) const { return (uint64_t)(t - a.l + 1u) * n - 1ull; }
    K2_HD uint32_t dec_range() const { return a.u - a.l + 1u; }
};
#define K2R_LE(c) ((uint64_t)(c) * range <= A)                       /* c <= target */

/* ------------------------------------------------------------------------------------------------ dense models
 * counts[card], total at [card]; rows are 16-byte aligned and padded to a multiple of four words. */
K2_HD uint32_t k2_rescale(uint32_t *m, uint32_t card) {               /* update_model :38-49 */
    uint32_t s = 0;
    for (uint32_t i = 0; i < card; i++) { const uint32_t c = (m[i] >> 1) + 1u; m[i] = c; s += c; }
    return s;
}
K2_HD uint32_t k2_cum_below(const uint32_t *m, uint32_t x) {          /* sum of m[0 .. x) */
    uint32_t s = 0, i = 0;
    for (; i + 4u <= x; i += 4u) { const K2U4 v = k2_ld4(m + i); s += v.x + v.y + v.z + v.w; }
    if (i < x) { const K2U4 v = k2_ld4(m + i); s += v.x + (i + 1u < x ? v.y : 0u) + (i + 2u < x ? v.z : 0u); }
    return s;
}
/* first x with cum(x + 1) > target */
K2_HD bool k2_find(const uint32_t *m, uint32_t card, uint64_t A, uint32_t range, uint32_t &x, uint32_t &lo, uint32_t &cnt) {
    uint32_t cum = 0;
    for (uint32_t i = 0; i < card; i += 4u) {
        const K2U4 v = k2_ld4(m + i);
        const uint32_t c1 = cum + v.x, c2 = c1 + (i + 1u < card ? v.y : 0u), c3 = c2 + (i + 2u < card ? v.z : 0u), c4 = c3 + (i + 3u < card ? v.w : 0u);
        if (!K2R_LE(c4)) {
            if (!K2R_LE(c1)) { x = i; lo = cum; cnt = v.x; }
            else if (!K2R_LE(c2)) { x = i + 1u; lo = c1; cnt = v.y; }
            else if (!K2R_LE(c3)) { x = i + 2u; lo = c2; cnt = v.z; }
            else { x = i + 3u; lo = c3; cnt = v.w; }
            return x < card;
        }
        cum = c4;
    }
    return false;
}
K2_HD void k2_update(uint32_t *m, uint32_t card, uint32_t step, uint32_t x, uint32_t cnt, uint32_t n) {
    m[x] = cnt + step;
    n += step;
    if (K2R_UNLIKELY(n >= CBCG_RESCALE)) n = k2_rescale(m, card);
    m[card] = n;
}
/* one symbol of a dense model: send_value_to_as / read_value_from_as + update_model */
template <int MODE>
K2_HD uint32_t k2_sym(K2Ac &ac, uint32_t *m, uint32_t card, uint32_t step, uint32_t x) {
    if (ac.err) return 0u;
    const uint32_t n = m[card];
    uint32_t lo, cnt;
    if (MODE == MODE_ENC) {
        if (K2R_UNLIKELY(x >= card)) { ac.err = CBCG_ERR_INPUT; return 0u; }           /* reference: assert :62 */
        lo = k2_cum_below(m, x); cnt = m[x];
        ac.encode(lo, cnt, n);
    } else {
        const uint64_t A = ac.dec_A(n); const uint32_t range = ac.dec_range();
        if (!k2_find(m, card, A, range, x, lo, cnt)) { ac.err = CBCG_ERR_CORRUPT; return 0u; }
        ac.decode_step(lo, cnt, n);
    }
    if (K2R_UNLIKELY(ac.err)) return 0u;
    k2_update(m, card, step, x, cnt, n);
    return x;
}

/* ------------------------------------------------------------------------------------------------ FLAG (sparse)
 * 65 536 symbols, all ones initially (src/sam_models.c:96-130): only the touched values are stored, ascending. */
template <int MODE>
K2_HD uint32_t k2_sym_flag(K2Ac &ac, WarpModels *M, uint32_t x) {
    if (ac.err) return 0u;
    const uint32_t used = M->flag_used, n = M->flag_n;
    uint32_t lo = 0, cnt = 1u, idx = 0; bool found = false;
    if (MODE == MODE_ENC) {
        if (x > 0xffffu) { ac.err = CBCG_ERR_INPUT; return 0u; }
        uint32_t extra = 0;
        for (idx = 0; idx < used; idx++) {
            const uint32_t k = M->flag_key[idx];
            if (k >= x) { if (k == x) { found = true; cnt = M->flag_cnt[idx]; } break; }
            extra += M->flag_cnt[idx] - 1u;
        }
        lo = x + extra;
        ac.encode(lo, cnt, n);
    } else {
        const uint64_t A = ac.dec_A(n); const uint32_t range = ac.dec_range();
        uint32_t extra = 0; bool done = false;
        for (idx = 0; idx < used; idx++) {
            const uint32_t k = M->flag_key[idx], c = M->flag_cnt[idx];
            const uint32_t start = k + extra;                          /* cumulative count at the start of value k */
            if (!K2R_LE(start)) break;                                 /* target lies before this touched value: an untouched one */
            if (!K2R_LE(start + c)) { x = k; lo = start; cnt = c; found = true; done = true; break; }
            extra += c - 1u;
        }
        if (!done) { const uint32_t target = ac_target(ac.a, ac.t, n); x = target - extra; lo = target; cnt = 1u; }
        if (x > 0xffffu) { ac.err = CBCG_ERR_CORRUPT; return 0u; }
        ac.decode_step(lo, cnt, n);
    }
    if (K2R_UNLIKELY(ac.err)) return 0u;
    uint32_t nused = used;
    if (found) M->flag_cnt[idx] = cnt + 8u;
    else {
        if (K2R_UNLIKELY(used >= FLAG_CAP)) return x;                     /* rule F1 (cbcg_format.h): coded at count 1, model unchanged */
        for (uint32_t j = used; j > idx; j--) { M->flag_key[j] = M->flag_key[j - 1u]; M->flag_cnt[j] = M->flag_cnt[j - 1u]; }
        M->flag_key[idx] = x; M->flag_cnt[idx] = 1u + 8u;
        nused = used + 1u; M->flag_used = nused;
    }
    uint32_t nn = n + 8u;
    if (K2R_UNLIKELY(nn >= CBCG_RESCALE)) nn = k2_rescale(M->flag_cnt, nused) + (65536u - nused);
    M->flag_n = nn;
    return x;
}

/* ------------------------------------------------------------------------------------------------ roles
 * Common: the block's workspace pieces (ws_layout order: pos_cnt | pos_val | pos_alpha | var_hash | var_rows). */
struct K2Block {
    const CoderParams *P; BlockDesc *B; uint32_t b;        /* b: absolute block index */
    WarpModels *M;                                           /* the block's image of the small models (fin) */
    WsLayout w; uint8_t *ws;
    SnapView snap;
    K2_HD void bind(const CoderParams &p, uint32_t block) {
        P = &p; b = block; B = &p.blocks[block];
        M = reinterpret_cast<WarpModels *>(p.fin + (uint64_t)block * fin_stride_dev());
        w = ws_layout(p.L, B->n_reads, B->n_edits, 0, 1);
        ws = p.ws + B->ws_off;
        snap = SnapView(p.snap, p.L);
    }
    K2_HD uint8_t *sub_out(uint32_t q) const {               /* encoder: scratch region of substream q */
        uint64_t o = B->payload_off;
        for (uint32_t j = 0; j < q; j++) o += k2_sub_cap(j, B->n_reads, B->n_edits);
        return P->payload + o;
    }
    K2_HD const uint8_t *sub_in(uint32_t q) const {          /* decoder: substream q in the compact payload */
        uint64_t o = B->payload_off;
        for (uint32_t j = 0; j < q; j++) o += B->sub_bytes[j];
        return P->payload + o;
    }
};
/* copy a piece of the snapshot's small-model image into the block's */
K2_HD void k2_copy_words(uint32_t *dst, const uint32_t *src, uint32_t n) { for (uint32_t i = 0; i < n; i++) dst[i] = src[i]; }

/* ---- substream A: POS through the growing alphabet (compress_pos :113-159, compress_pos_alpha :75-108) */
template <int MODE>
K2_HD int k2_role_pos(const CoderParams &P, uint32_t block, uint64_t *err_item) {
    K2Block K; K.bind(P, block);
    BlockDesc &B = *K.B;
    uint32_t *cntv = reinterpret_cast<uint32_t *>(K.ws + K.w.pos_cnt), *valv = reinterpret_cast<uint32_t *>(K.ws + K.w.pos_val);
    uint32_t *pa = reinterpret_cast<uint32_t *>(K.ws + K.w.pos_alpha);
    uint32_t card = K.snap.pos_hdr()[0], n = K.snap.pos_hdr()[1];
    if (card > K.w.pos_cap) return CBCG_ERR_INTERNAL;
    for (uint32_t i = 0; i < card; i++) { valv[i] = K.snap.pos_val()[i]; cntv[i] = K.snap.pos_cnt()[i]; }
    bool pa_init = false;
    K2Ac ac;
    if (MODE == MODE_ENC) ac.init_enc(K.sub_out(CBCG_SUB_POS), (uint32_t)k2_sub_cap(CBCG_SUB_POS, B.n_reads, B.n_edits));
    else ac.init_dec(K.sub_in(CBCG_SUB_POS), B.sub_bytes[CBCG_SUB_POS]);
    uint32_t prev_pos = B.base_pos;
    const uint64_t r0 = B.first_read;
    uint32_t i = 0;
    for (; i < B.n_reads; i++) {
        uint32_t x = 0, pos = 0, slot = 0, lo = 0, cnt = 0;
        if (MODE == MODE_ENC) {
            pos = P.recs[r0 + i].pos;
            if (pos == 0u || pos < prev_pos || pos - prev_pos + 1u > CBCG_MAX_POS_X) { ac.err = CBCG_ERR_INPUT; break; }
            x = pos - prev_pos + 1u;
            for (slot = 1; slot < card; slot++) { if (valv[slot] == x) break; }
            if (slot < card) { lo = k2_cum_below(cntv, slot); cnt = cntv[slot]; }
            else { slot = 0; lo = 0; cnt = cntv[0]; }
            ac.encode(lo, cnt, n);
        } else {
            const uint64_t A = ac.dec_A(n); const uint32_t range = ac.dec_range();
            if (!k2_find(cntv, card, A, range, slot, lo, cnt)) { ac.err = CBCG_ERR_CORRUPT; break; }
            ac.decode_step(lo, cnt, n);
            x = valv[slot];
        }
        if (ac.err) break;
        /* update_model, step 10 */
        cntv[slot] = cnt + 10u; n += 10u;
        if (K2R_UNLIKELY(n >= CBCG_RESCALE)) n = k2_rescale(cntv, card);
        if (slot == 0u) {                                      /* escape: the value itself, 4 bytes MSB first, then a new slot */
            if (!pa_init) {
                k2_copy_words(pa, K.snap.pos_alpha(), 4u * PA_STRIDE);
                pa_init = true;
            }
            uint32_t acc = 0;
            for (uint32_t k = 0; k < 4u; k++) {
                const uint32_t y = k2_sym<MODE>(ac, pa + k * PA_STRIDE, 256u, 10u, (x >> (24u - 8u * k)) & 0xffu);
                acc |= y << (24u - 8u * k);
            }
            if (ac.err) break;
            if (MODE == MODE_DEC) x = acc;
            if (card >= K.w.pos_cap) { ac.err = CBCG_ERR_INTERNAL; break; }
            valv[card] = x; cntv[card] = 10u; card++; n += 10u;              /* appended with count 0, then updated (:147-153) */
            if (K2R_UNLIKELY(n >= CBCG_RESCALE)) n = k2_rescale(cntv, card);
        }
        if (MODE == MODE_DEC) {
            if (x == 0u) { ac.err = CBCG_ERR_CORRUPT; break; }
            pos = prev_pos + x - 1u;
            if (pos == 0u) { ac.err = CBCG_ERR_CORRUPT; break; }
            P.recs[r0 + i].pos = pos;
            P.chr[r0 + i] = B.chr;
        }
        prev_pos = pos;
    }
    if (ac.err) { *err_item = ((uint64_t)block << 20) | (i & 0xfffffu); return ac.err; }
    if (MODE == MODE_ENC) { B.sub_bytes[CBCG_SUB_POS] = ac.finish_short(); if (ac.err) { *err_item = (uint64_t)block << 20; return ac.err; } }
    B.pos_card = card; B.pa_touched = pa_init ? 1u : 0u;
    k2_add_u32(&B.n_symbols, ac.nsym);
    return 0;
}

/* ---- substream B: length byte 0 (variable-length containers) and FLAG (compress_read :29-33, compress_flag :50-70) */
template <int MODE>
K2_HD int k2_role_flag(const CoderParams &P, uint32_t block, uint64_t *err_item) {
    K2Block K; K.bind(P, block);
    BlockDesc &B = *K.B;
    const WarpModels *S = reinterpret_cast<const WarpModels *>(K.snap.small());
    WarpModels *M = K.M;
    const bool fixed = P.fixed_len != 0;
    k2_copy_words(M->rlen0, S->rlen0, 256u);                   /* with same_ref / rlenk: never coded here, but the merge reads the whole image */
    k2_copy_words(M->same_ref, S->same_ref, 4u); k2_copy_words(&M->rlenk[0][0], &S->rlenk[0][0], 6u);
    { const uint32_t used = S->flag_used; for (uint32_t i = 0; i < used; i++) { M->flag_key[i] = S->flag_key[i]; M->flag_cnt[i] = S->flag_cnt[i]; } M->flag_used = used; M->flag_n = S->flag_n; }
    K2Ac ac;
    if (MODE == MODE_ENC) ac.init_enc(K.sub_out(CBCG_SUB_FLAG), (uint32_t)k2_sub_cap(CBCG_SUB_FLAG, B.n_reads, B.n_edits));
    else ac.init_dec(K.sub_in(CBCG_SUB_FLAG), B.sub_bytes[CBCG_SUB_FLAG]);
    const uint64_t r0 = B.first_read;
    uint32_t i = 0;
    for (; i < B.n_reads; i++) {
        uint32_t len = P.L, flag = 0;
        if (MODE == MODE_ENC) {
            const cbcg_read_rec rec = P.recs[r0 + i];
            len = rec.len; flag = rec.flag;
            if (len == 0u || len > CBCG_MAX_READ_LEN || (fixed && len != P.L)) { ac.err = CBCG_ERR_INPUT; break; }
        }
        if (!fixed) len = k2_sym<MODE>(ac, M->rlen0, 255u, 10u, len & 0xffu);
        flag = k2_sym_flag<MODE>(ac, M, flag);
        if (ac.err) break;
        if (MODE == MODE_DEC) {
            if (len == 0u || len > CBCG_MAX_READ_LEN) { ac.err = CBCG_ERR_CORRUPT; break; }
            P.recs[r0 + i].flag = (uint16_t)flag; P.recs[r0 + i].len = (uint16_t)len;
        }
    }
    if (ac.err) { *err_item = ((uint64_t)block << 20) | (i & 0xfffffu); return ac.err; }
    if (MODE == MODE_ENC) { B.sub_bytes[CBCG_SUB_FLAG] = ac.finish_short(); if (ac.err) { *err_item = (uint64_t)block << 20; return ac.err; } }
    k2_add_u32(&B.n_symbols, ac.nsym);
    return 0;
}

/* ---- substream C: match bit, SNP count, indel counts (compress_match :164-188, compress_snps / compress_indels :193-228,
 * the counts of compress_edits :557-565) */
template <int MODE>
K2_HD int k2_role_counts(const CoderParams &P, uint32_t block, uint64_t *err_item) {
    K2Block K; K.bind(P, block);
    BlockDesc &B = *K.B;
    const WarpModels *S = reinterpret_cast<const WarpModels *>(K.snap.small());
    WarpModels *M = K.M;
    const uint32_t L = P.L;
    k2_copy_words(M->snps, S->snps, 256u); k2_copy_words(M->indels, S->indels, 256u);
    k2_copy_words(&M->match[0][0], &S->match[0][0], 16u);
    K2Ac ac;
    if (MODE == MODE_ENC) ac.init_enc(K.sub_out(CBCG_SUB_COUNTS), (uint32_t)k2_sub_cap(CBCG_SUB_COUNTS, B.n_reads, B.n_edits));
    else ac.init_dec(K.sub_in(CBCG_SUB_COUNTS), B.sub_bytes[CBCG_SUB_COUNTS]);
    const uint64_t r0 = B.first_read;
    uint32_t prev_pos = B.base_pos, prev_m = 0u;
    uint64_t edits_left = B.n_edits;                             /* decoder: room in the block's edit range */
    uint32_t i = 0;
    for (; i < B.n_reads; i++) {
        const cbcg_read_rec rec = P.recs[r0 + i];                /* decoder: pos, flag, len come from the substreams A and B */
        const uint32_t samepos = rec.pos == prev_pos ? 1u : 0u;  /* deltaP == 1 (:170) */
        prev_pos = rec.pos;
        uint32_t match = rec.match, ns = rec.n_snps, nd = rec.n_dels, ni = rec.n_ins;
        match = k2_sym<MODE>(ac, M->match[(samepos << 1) | prev_m], 2u, 1u, match);
        if (ac.err) break;
        prev_m = match;
        if (!match) {
            uint32_t x = ((nd | ni) == 0u) ? ns : 0u;
            x = k2_sym<MODE>(ac, M->snps, L, 10u, x);
            if (MODE == MODE_DEC) { ns = x; nd = ni = 0; }
            if (!ac.err && (MODE == MODE_DEC ? x == 0u : (nd | ni) != 0u)) {   /* :560-565; the decoder takes a zero count as "indels follow" (:383-391) */
                ns = k2_sym<MODE>(ac, M->indels, L, 16u, ns);
                nd = k2_sym<MODE>(ac, M->indels, L, 16u, nd);
                ni = k2_sym<MODE>(ac, M->indels, L, 16u, ni);
            }
            if (ac.err) break;
            if (MODE == MODE_DEC) {
                if (ni > rec.len || ns > 255u || nd > 255u || ni > 255u) { ac.err = CBCG_ERR_CORRUPT; break; }
                if ((uint64_t)(ns + nd + ni) > edits_left) { ac.err = CBCG_ERR_CAPACITY; break; }
                edits_left -= ns + nd + ni;
            }
        } else if (MODE == MODE_DEC) { ns = nd = ni = 0; }
        if (MODE == MODE_DEC) {
            cbcg_read_rec *o = &P.recs[r0 + i];
            o->match = (uint8_t)match; o->n_snps = (uint8_t)ns; o->n_dels = (uint8_t)nd; o->n_ins = (uint8_t)ni;
        }
    }
    if (ac.err) { *err_item = ((uint64_t)block << 20) | (i & 0xfffffu); return ac.err; }
    if (MODE == MODE_ENC) { B.sub_bytes[CBCG_SUB_COUNTS] = ac.finish_short(); if (ac.err) { *err_item = (uint64_t)block << 20; return ac.err; } }
    k2_add_u32(&B.n_symbols, ac.nsym);
    return 0;
}

/* ---- substream D: edit positions through the var rows, bases through chars (:568-600; compute_delta_to_first_snp
 * :703-718). var rows: created on first touch in the block's arena behind a hash; a first touch is DEFERRED -- the
 * symbol is coded straight from the snapshot's row (read only; an all-ones row stands in for contexts the snapshot
 * has not seen), the hash slot notes "touched once, symbol x" -- and the row is only built, with that first update
 * applied, when the context comes back (most contexts are touched once per block). */
struct K2Var {
    uint64_t *hash; uint32_t mask; uint32_t *rows; uint32_t n_rows, rows_cap, Lp, L;
    SnapView snap;
    bool ro; uint32_t defer_idx, defer_key;
    K2_HD const uint32_t *snap_row(uint32_t ctx) const {
        const uint32_t w = snap.bitmap()[ctx >> 5];
        return ((w >> (ctx & 31u)) & 1u) ? snap.var_row(ctx) : snap.ones();
    }
    /* the row to code ctx with; ro set: it is the snapshot's (do not write; note_touch records the symbol) */
    K2_HD uint32_t *row(uint32_t ctx, int &err) {
        const uint32_t key = ctx + 1u;
        uint32_t idx = ((ctx * 0x9E3779B1u) >> 7) & mask;
        ro = false;
        for (uint32_t probes = 0; probes <= mask; probes++, idx = (idx + 1u) & mask) {
            const uint64_t s = hash[idx];
            const uint32_t k = (uint32_t)(s >> 32);
            if (k == key) {
                const uint32_t r = (uint32_t)s;
                if (!(r & VAR_DEFERRED)) return rows + (uint64_t)r * Lp;
                if (n_rows >= rows_cap) { err = CBCG_ERR_INTERNAL; return nullptr; }
                const uint32_t nr = n_rows++, x1 = r & 0xffffu;        /* second touch: build the row with the first touch applied */
                uint32_t *rw = rows + (uint64_t)nr * Lp;
                const uint32_t *src = snap_row(ctx);
                for (uint32_t i = 0; i <= L; i++) rw[i] = src[i];
                rw[x1] += 10u; rw[L] += 10u;
                hash[idx] = ((uint64_t)key << 32) | nr;
                return rw;
            }
            if (k == 0u) {
                defer_idx = idx; defer_key = key; ro = true;
                return const_cast<uint32_t *>(snap_row(ctx));
            }
        }
        err = CBCG_ERR_INTERNAL;
        return nullptr;
    }
    /* update_model (step 10) of the row `m` returned by row() for symbol x with count cnt and total n */
    K2_HD void update(uint32_t *m, uint32_t x, uint32_t cnt, uint32_t n, int &err) {
        if (!ro) { k2_update(m, L, 10u, x, cnt, n); return; }
        ro = false;
        if (K2R_LIKELY(n + 10u < CBCG_RESCALE)) { hash[defer_idx] = ((uint64_t)defer_key << 32) | VAR_DEFERRED | x; return; }
        if (n_rows >= rows_cap) { err = CBCG_ERR_INTERNAL; return; }                  /* the touch rescales the row: build it after all */
        const uint32_t nr = n_rows++;
        uint32_t *rw = rows + (uint64_t)nr * Lp;
        for (uint32_t i = 0; i <= L; i++) rw[i] = m[i];
        rw[x] += 10u;
        rw[L] = k2_rescale(rw, L);
        hash[defer_idx] = ((uint64_t)defer_key << 32) | nr;
    }
};
template <int MODE>
K2_HD uint32_t k2_sym_var(K2Ac &ac, K2Var &V, uint32_t ctx, uint32_t x) {
    if (ac.err) return 0u;
    if (ctx >= CBCG_VAR_CONTEXTS) { ac.err = (MODE == MODE_ENC) ? CBCG_ERR_INPUT : CBCG_ERR_CORRUPT; return 0u; }
    uint32_t *m = V.row(ctx, ac.err);
    if (!m) return 0u;
    const uint32_t L = V.L, n = m[L];
    uint32_t lo, cnt;
    if (MODE == MODE_ENC) {
        if (K2R_UNLIKELY(x >= L)) { ac.err = CBCG_ERR_INPUT; return 0u; }
        lo = k2_cum_below(m, x); cnt = m[x];
        ac.encode(lo, cnt, n);
    } else {
        const uint64_t A = ac.dec_A(n); const uint32_t range = ac.dec_range();
        if (!k2_find(m, L, A, range, x, lo, cnt)) { ac.err = CBCG_ERR_CORRUPT; return 0u; }
        ac.decode_step(lo, cnt, n);
    }
    if (K2R_UNLIKELY(ac.err)) return 0u;
    V.update(m, x, cnt, n, ac.err);
    return x;
}

/* snpInRef[] (a 300 MB byte map in the reference, include/read_compression.h:28): reads are position-sorted, so only
 * [pos - 1, pos + L) is ever consulted: a 1024-bit ring, word (p >> 5) & 31. */
struct K2Ring {
    uint32_t w[32]; uint32_t word0;                            /* covers bit positions [word0 * 32, word0 * 32 + 1024) */
    K2_HD void reset() { for (uint32_t i = 0; i < 32u; i++) w[i] = 0u; word0 = 0u; }
    K2_HD void advance(uint32_t pos) {                          /* the window must start at or below pos - 1 */
        const uint32_t nw = (pos - 1u) >> 5;
        if (nw > word0) {
            const uint32_t adv = nw - word0;
            if (adv >= 32u) { for (uint32_t i = 0; i < 32u; i++) w[i] = 0u; }
            else for (uint32_t j = 0; j < adv; j++) w[(word0 + j) & 31u] = 0u;   /* words that rotate out and back in */
            word0 = nw;
        }
    }
    K2_HD void set(uint32_t p) { if ((p >> 5) - word0 < 32u) w[(p >> 5) & 31u] |= 1u << (p & 31u); }
    /* distance from s to the first marked site in [s, e), else `none` (compute_delta_to_first_snp) */
    K2_HD uint32_t first(uint32_t s, uint32_t e, uint32_t none) const {
        if (e <= s) return none;
        for (uint32_t wd = s >> 5; (wd << 5) < e; wd++) {
            if (wd - word0 >= 32u) break;
            uint32_t bits = w[wd & 31u];
            if (wd == (s >> 5)) bits &= 0xffffffffu << (s & 31u);
            if (((wd + 1u) << 5) > e) bits &= (e & 31u) ? ((1u << (e & 31u)) - 1u) : 0xffffffffu;
            if (bits) {
#ifdef __CUDA_ARCH__
                return (wd << 5) + (uint32_t)__ffs((int)bits) - 1u - s;
#else
                return (wd << 5) + (uint32_t)__builtin_ctz(bits) - s;
#endif
            }
        }
        return none;
    }
};

template <int MODE>
K2_HD int k2_role_edits(const CoderParams &P, uint32_t block, uint64_t *err_item) {
    K2Block K; K.bind(P, block);
    BlockDesc &B = *K.B;
    const WarpModels *S = reinterpret_cast<const WarpModels *>(K.snap.small());
    WarpModels *M = K.M;
    k2_copy_words(&M->chars[0][0], &S->chars[0][0], 48u);
    K2Var V;
    V.hash = reinterpret_cast<uint64_t *>(K.ws + K.w.var_hash); V.mask = K.w.hash_cap - 1u;
    V.rows = reinterpret_cast<uint32_t *>(K.ws + K.w.var_rows); V.n_rows = 0; V.rows_cap = K.w.rows_cap; V.Lp = K.w.Lp; V.L = P.L;
    V.snap = K.snap; V.ro = false; V.defer_idx = 0; V.defer_key = 0;
    for (uint32_t i = 0; i <= V.mask; i++) V.hash[i] = 0ull;
    K2Ring ring; ring.reset();
    K2Ac ac;
    if (MODE == MODE_ENC) ac.init_enc(K.sub_out(CBCG_SUB_EDITS), (uint32_t)k2_sub_cap(CBCG_SUB_EDITS, B.n_reads, B.n_edits));
    else ac.init_dec(K.sub_in(CBCG_SUB_EDITS), B.sub_bytes[CBCG_SUB_EDITS]);
    const uint64_t r0 = B.first_read;
    const uint8_t *ref = nullptr; uint64_t ref_len = 0;
    if (MODE == MODE_DEC) {
        if (B.chr >= P.genome.n_chr) { *err_item = (uint64_t)block << 20; return CBCG_ERR_NO_REFERENCE; }
        ref = P.genome.bases + P.genome.chr_off[B.chr]; ref_len = P.genome.chr_len[B.chr];
    }
    uint64_t e_cursor = B.edit_base;
    uint16_t cumdel[256];
    uint32_t i = 0;
    for (; i < B.n_reads; i++) {
        const cbcg_read_rec rec = P.recs[r0 + i];
        const uint32_t pos = rec.pos, len = rec.len, strand = ((uint32_t)rec.flag >> 4) & 1u;     /* :57-60 */
        ring.advance(pos);
        if (MODE == MODE_DEC) P.recs[r0 + i].edit_off = (uint32_t)e_cursor;
        if (rec.match) continue;
        const uint32_t nd = rec.n_dels, ns = rec.n_snps, ni = rec.n_ins;
        const uint16_t *e_in = P.edits + rec.edit_off;          /* encoder */
        uint16_t *e_out = P.edits + e_cursor;                    /* decoder */
        uint32_t prev = 0, ne = 0;
        for (uint32_t k = 0; k < nd; k++) {                       /* deletions (:568-572) */
            const uint32_t d = k2_sym_var<MODE>(ac, V, (prev << 1) | strand, MODE == MODE_ENC ? CBCG_EDIT_DELTA(e_in[k]) : 0u);
            prev += d;
            if (MODE == MODE_DEC) { e_out[ne] = CBCG_EDIT(d, 0, 0); cumdel[k] = (uint16_t)(prev < 0xffffu ? prev : 0xffffu); }
            ne++;
        }
        prev = 0;
        for (uint32_t k = 0; k < ns && !ac.err; k++) {            /* SNPs (:573-593) */
            const uint32_t ed = MODE == MODE_ENC ? e_in[nd + k] : 0u;
            const uint32_t delta = ring.first(pos - 1u + prev, (prev < len) ? pos - 1u + len : pos - 1u + prev, len + 2u);
            const uint32_t ctx = (((delta << CBCG_BITS_DELTA) + prev) << 1) | strand;
            const uint32_t p = k2_sym_var<MODE>(ac, V, ctx, CBCG_EDIT_DELTA(ed));
            if (ac.err) break;
            const uint32_t idx = prev + p;                        /* index in the insertion-free read */
            prev += p + 1u;
            ring.set(pos + prev - 2u);                            /* :589 */
            uint32_t refb;
            if (MODE == MODE_DEC) {
                uint32_t skipped = 0;                             /* deletions at or before idx (:426-437) */
                while (skipped < nd && cumdel[skipped] <= idx) skipped++;
                const uint64_t ri = (uint64_t)pos - 1u + idx + skipped;
                refb = k2_base_code(ri < ref_len ? (uint32_t)ref[ri] : 0u);
            } else refb = CBCG_EDIT_REFB(ed);
            if (refb > 5u) { ac.err = CBCG_ERR_INPUT; break; }
            const uint32_t tgt = k2_sym<MODE>(ac, M->chars[refb], 5u, 8u, CBCG_EDIT_TARGET(ed));
            if (MODE == MODE_DEC) e_out[ne] = CBCG_EDIT(p, tgt, refb);
            ne++;
        }
        prev = 0;
        for (uint32_t k = 0; k < ni && !ac.err; k++) {            /* insertions (:594-600) */
            const uint32_t ed = MODE == MODE_ENC ? e_in[nd + ns + k] : 0u;
            const uint32_t p = k2_sym_var<MODE>(ac, V, (prev << 1) | strand, CBCG_EDIT_DELTA(ed));
            prev += p;
            const uint32_t tgt = k2_sym<MODE>(ac, M->chars[CBCG_BP_O], 5u, 8u, CBCG_EDIT_TARGET(ed));
            if (MODE == MODE_DEC) e_out[ne] = CBCG_EDIT(p, tgt, CBCG_BP_O);
            ne++;
        }
        if (ac.err) break;
        e_cursor += ne;
    }
    if (ac.err) { *err_item = ((uint64_t)block << 20) | (i & 0xfffffu); return ac.err; }
    if (MODE == MODE_ENC) { B.sub_bytes[CBCG_SUB_EDITS] = ac.finish_short(); if (ac.err) { *err_item = (uint64_t)block << 20; return ac.err; } }
    if (MODE == MODE_DEC && e_cursor - B.edit_base != B.n_edits) { *err_item = (uint64_t)block << 20; return CBCG_ERR_CORRUPT; }   /* the index said otherwise */
    B.n_rows = V.n_rows;
    k2_add_u32(&B.n_symbols, ac.nsym);
    return 0;
}

/* substream q of one block */
template <int MODE>
K2_HD int k2_run_role(const CoderParams &P, uint32_t q, uint32_t block, uint64_t *err_item) {
    switch (q) {
        case CBCG_SUB_POS:    return k2_role_pos<MODE>(P, block, err_item);
        case CBCG_SUB_FLAG:   return k2_role_flag<MODE>(P, block, err_item);
        case CBCG_SUB_COUNTS: return k2_role_counts<MODE>(P, block, err_item);
        default:              return k2_role_edits<MODE>(P, block, err_item);
    }
}

/* ------------------------------------------------------------------------------------------------
 * S_{-1}: the reference's initial model state in snapshot form (sam_models.c:56-411, :562-586): what the blocks of
 * generation 0 -- and every block of a gen_mode 0 container -- start from. One thread. */
K2_HD void k2_snapshot_init(uint8_t *snap, uint32_t L) {
    const SnapLayout l = snap_layout(L);
    WarpModels *M = reinterpret_cast<WarpModels *>(snap + l.small);
    uint32_t *w = reinterpret_cast<uint32_t *>(M);
    for (uint32_t i = 0; i < (uint32_t)(sizeof(WarpModels) / 4u); i++) w[i] = 0u;
    for (uint32_t i = 0; i < L; i++) { M->snps[i] = 1u; M->indels[i] = 1u; }
    M->snps[L] = L; M->indels[L] = L;
    for (uint32_t i = 0; i < 255u; i++) M->rlen0[i] = 1u;
    M->rlen0[255] = 255u;
    for (uint32_t r = 0; r < 6u; r++) {                       /* initialize_stream_model_chars :350-411 */
        uint32_t n = 0;
        for (uint32_t i = 0; i < 4u; i++) { const uint32_t c = (i == r) ? 0u : 8u; M->chars[r][i] = c; n += c; }
        M->chars[r][4] = 1u; n += 1u;
        if (r < 4u) {
            const uint32_t f0 = (r == 0u || r == 3u) ? 1u : 0u, f1 = (r == 0u || r == 3u) ? 2u : 3u;
            M->chars[r][f0] += 8u; M->chars[r][f1] += 8u; n += 16u;
        }
        M->chars[r][5] = n;
    }
    for (uint32_t c = 0; c < 4u; c++) { M->match[c][0] = 1u; M->match[c][1] = 1u; M->match[c][2] = 2u; }
    M->same_ref[0] = 1u; M->same_ref[1] = 1u; M->same_ref[2] = 2u;
    for (uint32_t k = 0; k < 3u; k++) { M->rlenk[k][0] = 1u; M->rlenk[k][1] = 255u; }
    M->flag_used = 0u; M->flag_n = 65536u;
    uint32_t *hdr = reinterpret_cast<uint32_t *>(snap + l.pos_hdr);
    uint32_t *pv = reinterpret_cast<uint32_t *>(snap + l.pos_val), *pc = reinterpret_cast<uint32_t *>(snap + l.pos_cnt);
    hdr[0] = 1u; hdr[1] = 1u; hdr[2] = 0u; hdr[3] = 0u; pv[0] = 0u; pc[0] = 1u;      /* escape only (:132-162) */
    uint32_t *pa = reinterpret_cast<uint32_t *>(snap + l.pos_alpha);
    for (uint32_t k = 0; k < 4u; k++) { for (uint32_t i = 0; i < 256u; i++) pa[k * PA_STRIDE + i] = 1u; pa[k * PA_STRIDE + 256u] = 256u; }
    uint32_t *bm = reinterpret_cast<uint32_t *>(snap + l.bitmap);
    for (uint32_t i = 0; i < 2048u; i++) bm[i] = 0u;
    uint32_t *ones = reinterpret_cast<uint32_t *>(snap + l.ones);
    for (uint32_t i = 0; i < L; i++) ones[i] = 1u;
    ones[L] = L;
}
