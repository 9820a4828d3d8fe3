/*
 * oracle/cbc_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (see cbc_oracle.h).
 *
 * Plain-C restatement of the reference's aligned-read coding path, written from the
 * reference's behaviour (citations are reference file:line), not copied from it.
 * Pinned against the unmodified reference built into oracle/_ref/ (byte-identical
 * streams, identical symbol traces): tests/test_oracle_vs_reference.py, tests/golden/.
 */
#include "cbc_oracle.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ctype.h>

/* ------------------------------------------------------------------ growable buffer */

static int buf_reserve(cbco_buf *b, uint64_t extra) {
    if (b->size + extra <= b->cap) return 0;
    uint64_t cap = b->cap ? b->cap : 4096;
    while (cap < b->size + extra) cap *= 2;
    uint8_t *p = (uint8_t *)realloc(b->data, cap);
    if (!p) return -1;
    b->data = p; b->cap = cap;
    return 0;
}
static void buf_put(cbco_buf *b, const void *src, uint64_t n) {
    if (buf_reserve(b, n)) abort();
    memcpy(b->data + b->size, src, n);
    b->size += n;
}
static void buf_put_u32(cbco_buf *b, uint32_t v) { buf_put(b, &v, 4); }
static void buf_put_u64(cbco_buf *b, uint64_t v) { buf_put(b, &v, 8); }
void cbco_buf_free(cbco_buf *b) { free(b->data); b->data = NULL; b->size = b->cap = 0; }

/* ------------------------------------------------------------------ base helpers
 * char2basepair / basepair2char / bp_complement: src/sam_models.c:11-45 */
static int base_code(int c) {
    switch (c) { case 'A': return 0; case 'C': return 1; case 'G': return 2; case 'T': return 3; default: return 4; }
}
static int base_char(int b) {
    switch (b) { case 0: return 'A'; case 1: return 'C'; case 2: return 'G'; case 3: return 'T'; default: return 'N'; }
}

/* ------------------------------------------------------------------ bit stream
 * MSB-first bit packer: stream_write_bit / stream_finish_byte,
 * src/Arithmetic_stream.c:155-194. The reader returns zeros past the end, which is what
 * the reference's zero-filled 4 MiB buffer gives (src/Arithmetic_stream.c:30,117). */
typedef struct { cbco_buf *out; uint32_t acc; uint32_t nbits; } bitw;
static void bw_bit(bitw *w, uint32_t bit) {
    w->acc = (w->acc << 1) | (bit & 1u);
    if (++w->nbits == 8) { uint8_t v = (uint8_t)w->acc; buf_put(w->out, &v, 1); w->acc = 0; w->nbits = 0; }
}
static void bw_finish(bitw *w) {
    /* stream_finish_byte always emits the byte in progress, even an empty one. */
    uint8_t v = (uint8_t)(w->acc << (8 - w->nbits));
    if (w->nbits == 0) v = 0;
    buf_put(w->out, &v, 1);
    w->acc = 0; w->nbits = 0;
}
typedef struct { const uint8_t *p; uint64_t len; uint64_t bitpos; } bitr;
static uint32_t br_bit(bitr *r) {
    uint64_t byte = r->bitpos >> 3;
    uint32_t v = 0;
    if (byte < r->len) v = (r->p[byte] >> (7 - (r->bitpos & 7))) & 1u;
    r->bitpos++;
    return v;
}

/* ------------------------------------------------------------------ arithmetic coder
 * src/Arithmetic_stream.c:245-454. */
typedef struct { uint32_t l, u, t; int32_t scale3; bitw w; bitr r; } acoder;

static void ac_init_enc(acoder *a, cbco_buf *out) {
    memset(a, 0, sizeof *a);
    a->l = 0; a->u = CBCG_AC_TOP; a->w.out = out;
}
static void ac_init_dec(acoder *a, const uint8_t *p, uint64_t len) {
    memset(a, 0, sizeof *a);
    a->l = 0; a->u = CBCG_AC_TOP; a->r.p = p; a->r.len = len;
    for (uint32_t i = 0; i < CBCG_AC_BITS; i++) a->t = (a->t << 1) | br_bit(&a->r);   /* :262 */
}
static int ac_cond(const acoder *a, int *e3) {
    uint32_t ml = a->l >> (CBCG_AC_BITS - 1), mu = a->u >> (CBCG_AC_BITS - 1);
    *e3 = 0;
    if (ml == mu) return 1;
    *e3 = ((a->l >> (CBCG_AC_BITS - 2)) == 1u && (a->u >> (CBCG_AC_BITS - 2)) == 2u);
    return 0;
}
/* arithmetic_encoder_step :274-345 -- u is computed from the old l, then l. */
static int ac_encode(acoder *a, uint32_t lo, uint32_t hi, uint32_t n) {
    if (!(lo < hi) || n == 0) return -1;             /* reference: assert :293 */
    uint64_t range = (uint64_t)a->u - a->l + 1;
    a->u = a->l + (uint32_t)((range * hi) / n) - 1;
    a->l = a->l + (uint32_t)((range * lo) / n);
    int e3, e12 = ac_cond(a, &e3);
    while (e12 || e3) {
        if (e12) {
            uint32_t msb = a->l >> (CBCG_AC_BITS - 1);
            bw_bit(&a->w, msb);
            a->l = (a->l & CBCG_AC_LOWMASK) << 1;
            a->u = ((a->u & CBCG_AC_LOWMASK) << 1) + 1;
            while (a->scale3 > 0) { bw_bit(&a->w, !msb); a->scale3--; }
        } else {
            a->scale3++;
            a->u = (((a->u << 1) & CBCG_AC_LOWMASK) | CBCG_AC_MSB) + 1;
            a->l = (a->l << 1) & CBCG_AC_LOWMASK;
        }
        e12 = ac_cond(a, &e3);
    }
    return 0;
}
/* encoder_last_step :348-364 */
static void ac_flush(acoder *a) {
    uint32_t msb = a->l >> (CBCG_AC_BITS - 1);
    bw_bit(&a->w, msb);
    while (a->scale3 > 0) { bw_bit(&a->w, !msb); a->scale3--; }
    for (int bit = (int)CBCG_AC_BITS - 2; bit >= 0; --bit) bw_bit(&a->w, a->l >> bit);
    bw_finish(&a->w);
}
/* Blocked containers (our format): the shortest tail that still decodes. After renormalisation
 * l < 2^25 <= u, so the value 2^25 ("1", the pending E3 bits as "0", then zeros) lies in [l, u]; the
 * decoder reads zeros past the end of a block, so only 1 + scale3 bits go out, padded to a byte. */
uint64_t cbco_debug_flush_bits = 0;        /* experiments: bits the short tails added beyond the coded bits */
static void ac_flush_short(acoder *a) {
    const uint64_t before = a->w.out->size * 8u + a->w.nbits;
    cbco_debug_flush_bits -= before;
    bw_bit(&a->w, 1);
    while (a->scale3 > 0) { bw_bit(&a->w, 0); a->scale3--; }
    if (a->w.nbits) bw_finish(&a->w);
    cbco_debug_flush_bits += a->w.out->size * 8u;
}
/* arithmetic_get_symbol_range :373-381 */
static uint32_t ac_target(const acoder *a, uint32_t n) {
    uint64_t range = (uint64_t)a->u - a->l + 1;
    uint64_t gap = (uint64_t)a->t - a->l + 1;
    return (uint32_t)((gap * n - 1) / range);
}
/* arithmetic_decoder_step :389-454 */
static void ac_decode(acoder *a, uint32_t lo, uint32_t hi, uint32_t n) {
    uint64_t range = (uint64_t)a->u - a->l + 1;
    a->u = a->l + (uint32_t)((range * hi) / n) - 1;
    a->l = a->l + (uint32_t)((range * lo) / n);
    int e3, e12 = ac_cond(a, &e3);
    while (e12 || e3) {
        if (e12) {
            a->l = (a->l & CBCG_AC_LOWMASK) << 1;
            a->u = ((a->u & CBCG_AC_LOWMASK) << 1) + 1;
            a->t = ((a->t & CBCG_AC_LOWMASK) << 1) + br_bit(&a->r);
        } else {
            a->l = (a->l << 1) & CBCG_AC_LOWMASK;
            a->u = (((a->u << 1) & CBCG_AC_LOWMASK) | CBCG_AC_MSB) + 1;
            a->t = (((a->t & CBCG_AC_LOWMASK) << 1) ^ CBCG_AC_MSB) + br_bit(&a->r);
        }
        e12 = ac_cond(a, &e3);
    }
}

/* ------------------------------------------------------------------ adaptive models
 * stream_model_t / update_model / send_value_to_as / read_value_from_as:
 * include/stream_model.h:16-27, src/stream_model.c:31-117. */
typedef struct { uint32_t *c; uint32_t card, step, n; } model;

static void model_ones(model *m, uint32_t card, uint32_t step) {
    m->c = (uint32_t *)malloc(sizeof(uint32_t) * (card ? card : 1));
    for (uint32_t i = 0; i < card; i++) m->c[i] = 1;
    m->card = card; m->step = step; m->n = card;
}
static void model_free(model *m) { free(m->c); m->c = NULL; }
static void model_update(model *m, uint32_t x) {
    m->c[x] += m->step; m->n += m->step;
    if (m->n >= CBCG_RESCALE) {
        m->n = 0;
        for (uint32_t i = 0; i < m->card; i++) { m->c[i] = (m->c[i] >> 1) + 1; m->n += m->c[i]; }
    }
}

/* The pos model grows: new symbols are appended with count 0 (src/sam_models.c:132-162,
 * src/read_compression.c:113-159). x -> slot lookup through a small hash map. */
typedef struct {
    model m; uint32_t cap; uint32_t *alpha;   /* alpha[slot] = x (slot 0 = escape) */
    uint32_t *hkey, *hval; uint32_t hcap, hcount;
} posmodel;

static void pos_hash_put(posmodel *p, uint32_t x, uint32_t slot);
static void pos_init(posmodel *p) {
    memset(p, 0, sizeof *p);
    p->cap = 1024;
    p->m.c = (uint32_t *)calloc(p->cap, sizeof(uint32_t));
    p->alpha = (uint32_t *)calloc(p->cap, sizeof(uint32_t));
    p->m.card = 1; p->m.c[0] = 1; p->m.n = 1; p->m.step = 10;
    p->hcap = 4096;
    p->hkey = (uint32_t *)malloc(sizeof(uint32_t) * p->hcap);
    p->hval = (uint32_t *)malloc(sizeof(uint32_t) * p->hcap);
    memset(p->hkey, 0xff, sizeof(uint32_t) * p->hcap);
}
static void pos_free(posmodel *p) { free(p->m.c); free(p->alpha); free(p->hkey); free(p->hval); }
static uint32_t pos_hash(uint32_t x) { x *= 0x9e3779b1u; return x ^ (x >> 15); }
static int pos_find(const posmodel *p, uint32_t x) {
    uint32_t s = pos_hash(x) & (p->hcap - 1);
    while (p->hkey[s] != 0xffffffffu) {
        if (p->hkey[s] == x) return (int)p->hval[s];
        s = (s + 1) & (p->hcap - 1);
    }
    return -1;
}
static void pos_hash_put(posmodel *p, uint32_t x, uint32_t slot) {
    if ((p->hcount + 1) * 2 > p->hcap) {
        uint32_t ocap = p->hcap, *ok = p->hkey, *ov = p->hval;
        p->hcap *= 2; p->hcount = 0;
        p->hkey = (uint32_t *)malloc(sizeof(uint32_t) * p->hcap);
        p->hval = (uint32_t *)malloc(sizeof(uint32_t) * p->hcap);
        memset(p->hkey, 0xff, sizeof(uint32_t) * p->hcap);
        for (uint32_t i = 0; i < ocap; i++) if (ok[i] != 0xffffffffu) pos_hash_put(p, ok[i], ov[i]);
        free(ok); free(ov);
    }
    uint32_t s = pos_hash(x) & (p->hcap - 1);
    while (p->hkey[s] != 0xffffffffu) s = (s + 1) & (p->hcap - 1);
    p->hkey[s] = x; p->hval[s] = slot; p->hcount++;
}
static uint32_t pos_append(posmodel *p, uint32_t x) {
    if (p->m.card == p->cap) {
        p->cap *= 2;
        p->m.c = (uint32_t *)realloc(p->m.c, sizeof(uint32_t) * p->cap);
        p->alpha = (uint32_t *)realloc(p->alpha, sizeof(uint32_t) * p->cap);
    }
    uint32_t slot = p->m.card++;
    p->m.c[slot] = 0; p->alpha[slot] = x;
    pos_hash_put(p, x, slot);
    return slot;
}

/* All models of one coder instance (alloc_read_models_t src/sam_models.c:562-586,
 * alloc_rname_models_t :611-620, initialize_stream_model_codebook :734-770). var rows
 * are created on first touch: their initial state is all-ones, so this is invisible. */
typedef struct models_s {
    uint32_t L;                 /* header read length: alphabet of snps/indels/var */
    model codebook[4], same_ref, rname[256], rlength[4], pos_alpha[4], flag, match[4], snps, indels, chars[6];
    model *var;                 /* CBCG_VAR_CONTEXTS lazily initialised rows (c == NULL: untouched) */
    posmodel pos;
    const struct models_s *base; /* primed blocks: untouched var rows are read from this snapshot (copy on first touch) */
    uint32_t flag_adapted;      /* FLAG values whose count is not the initial 1 (blocked containers adapt at most
                                   CBCG_FLAG_ADAPT_MAX of them: rules F1 / F2, cbcg_format.h) */
} models;

static void chars_init(model *m, int row) {
    /* initialize_stream_model_chars src/sam_models.c:350-411 */
    m->c = (uint32_t *)malloc(sizeof(uint32_t) * 5);
    m->card = 5; m->step = 8; m->n = 0;
    for (int i = 0; i < 4; i++) { m->c[i] = (i == row) ? 0 : 8; m->n += m->c[i]; }
    m->c[4] = 1; m->n++;
    static const int fav[4][2] = { {1, 2}, {0, 3}, {0, 3}, {1, 2} };
    if (row < 4) { m->c[fav[row][0]] += 8; m->c[fav[row][1]] += 8; m->n += 16; }
}
static void models_init(models *M, uint32_t L) {
    memset(M, 0, sizeof *M);
    M->L = L;
    for (int i = 0; i < 4; i++) model_ones(&M->codebook[i], 256, 1);
    model_ones(&M->same_ref, 2, 10);
    for (int i = 0; i < 256; i++) model_ones(&M->rname[i], 256, 10);
    for (int i = 0; i < 4; i++) model_ones(&M->rlength[i], 255, 10);
    for (int i = 0; i < 4; i++) model_ones(&M->pos_alpha[i], 256, 10);
    model_ones(&M->flag, 1u << 16, 8);
    for (int i = 0; i < 4; i++) model_ones(&M->match[i], 2, 1);
    model_ones(&M->snps, L, 10);
    model_ones(&M->indels, L, 16);
    for (int i = 0; i < 6; i++) chars_init(&M->chars[i], i);
    M->var = (model *)calloc(CBCG_VAR_CONTEXTS, sizeof(model));
    pos_init(&M->pos);
}
static void models_free(models *M) {
    for (int i = 0; i < 4; i++) { model_free(&M->codebook[i]); model_free(&M->rlength[i]); model_free(&M->pos_alpha[i]); model_free(&M->match[i]); }
    for (int i = 0; i < 256; i++) model_free(&M->rname[i]);
    for (int i = 0; i < 6; i++) model_free(&M->chars[i]);
    model_free(&M->same_ref); model_free(&M->flag); model_free(&M->snps); model_free(&M->indels);
    for (uint32_t i = 0; i < CBCG_VAR_CONTEXTS; i++) if (M->var[i].c) model_free(&M->var[i]);
    free(M->var);
    pos_free(&M->pos);
}
static model *model_of(models *M, uint32_t stream, uint32_t ctx);

/* ------------------------------------------------------------------ generation-primed blocks (our design)
 * A block of generation g starts from the snapshot S_{g-1} (S_{-1}: the reference's initial state) instead
 * of from scratch; S_g = S_{g-1} + sum over the blocks b of generation g of (final state of b - S_{g-1}),
 * count by count, clamped and rescaled like update_model does. The decoder rebuilds the same snapshots
 * from the blocks it has decoded, so blocks of one generation are independent of each other. */
static void model_clone(model *d, const model *s) {
    d->c = (uint32_t *)malloc(sizeof(uint32_t) * (s->card ? s->card : 1));
    memcpy(d->c, s->c, sizeof(uint32_t) * s->card);
    d->card = s->card; d->step = s->step; d->n = s->n;
}
static void pos_clone(posmodel *d, const posmodel *s) {
    memset(d, 0, sizeof *d);
    d->cap = s->cap;
    d->m.c = (uint32_t *)malloc(sizeof(uint32_t) * s->cap); memcpy(d->m.c, s->m.c, sizeof(uint32_t) * s->m.card);
    d->alpha = (uint32_t *)malloc(sizeof(uint32_t) * s->cap); memcpy(d->alpha, s->alpha, sizeof(uint32_t) * s->m.card);
    d->m.card = s->m.card; d->m.n = s->m.n; d->m.step = s->m.step;
    d->hcap = s->hcap; d->hcount = s->hcount;
    d->hkey = (uint32_t *)malloc(sizeof(uint32_t) * s->hcap); memcpy(d->hkey, s->hkey, sizeof(uint32_t) * s->hcap);
    d->hval = (uint32_t *)malloc(sizeof(uint32_t) * s->hcap); memcpy(d->hval, s->hval, sizeof(uint32_t) * s->hcap);
}
/* A block's working copy of a snapshot: small models copied, var rows copied on first touch. */
static void models_clone(models *M, const models *S) {
    memset(M, 0, sizeof *M);
    M->L = S->L;
    for (int i = 0; i < 4; i++) { model_clone(&M->codebook[i], &S->codebook[i]); model_clone(&M->rlength[i], &S->rlength[i]);
                                  model_clone(&M->pos_alpha[i], &S->pos_alpha[i]); model_clone(&M->match[i], &S->match[i]); }
    for (int i = 0; i < 256; i++) model_clone(&M->rname[i], &S->rname[i]);
    for (int i = 0; i < 6; i++) model_clone(&M->chars[i], &S->chars[i]);
    model_clone(&M->same_ref, &S->same_ref); model_clone(&M->flag, &S->flag);
    model_clone(&M->snps, &S->snps); model_clone(&M->indels, &S->indels);
    M->var = (model *)calloc(CBCG_VAR_CONTEXTS, sizeof(model));
    pos_clone(&M->pos, &S->pos);
    M->base = S;
    M->flag_adapted = S->flag_adapted;
}
/* acc += (fin - prev), wrapping 32-bit (exact as long as the true sum stays inside int32). */
static void merge_model(model *acc, const model *fin, const model *prev) {
    for (uint32_t i = 0; i < acc->card; i++) acc->c[i] += fin->c[i] - prev->c[i];
}
static void merge_block(models *acc, const models *fin, const models *prev) {
    for (int i = 0; i < 4; i++) { merge_model(&acc->rlength[i], &fin->rlength[i], &prev->rlength[i]);
                                  merge_model(&acc->pos_alpha[i], &fin->pos_alpha[i], &prev->pos_alpha[i]);
                                  merge_model(&acc->match[i], &fin->match[i], &prev->match[i]); }
    for (int i = 0; i < 6; i++) merge_model(&acc->chars[i], &fin->chars[i], &prev->chars[i]);
    merge_model(&acc->same_ref, &fin->same_ref, &prev->same_ref);
    merge_model(&acc->flag, &fin->flag, &prev->flag);
    merge_model(&acc->snps, &fin->snps, &prev->snps);
    merge_model(&acc->indels, &fin->indels, &prev->indels);
    for (uint32_t ctx = 0; ctx < CBCG_VAR_CONTEXTS; ctx++) {
        if (!fin->var[ctx].c) continue;                       /* untouched by the block */
        model *a = model_of(acc, CBCG_S_VAR, ctx);            /* materialises acc's copy of the snapshot row */
        const model *f = &fin->var[ctx];
        if (prev->var[ctx].c) for (uint32_t i = 0; i < a->card; i++) a->c[i] += f->c[i] - prev->var[ctx].c[i];
        else for (uint32_t i = 0; i < a->card; i++) a->c[i] += f->c[i] - 1u;
    }
    /* pos: values new to the snapshot are appended in block order, then order of appearance */
    for (uint32_t s = 0; s < fin->pos.m.card; s++) {
        uint32_t x = fin->pos.alpha[s];
        int ps = (s == 0) ? 0 : pos_find(&prev->pos, x);
        uint32_t before = (ps >= 0) ? prev->pos.m.c[ps] : 0u;
        int as = (s == 0) ? 0 : pos_find(&acc->pos, x);
        if (as < 0) {
            if (acc->pos.m.card >= CBCG_SNAP_POS_MAX) continue;   /* snapshot alphabet is capped; the value stays block-local */
            as = (int)pos_append(&acc->pos, x);
        }
        acc->pos.m.c[as] += fin->pos.m.c[s] - before;
    }
}
static void finish_model(model *m, const model *prev, uint32_t prev_card) {
    uint32_t n = 0;
    for (uint32_t i = 0; i < m->card; i++) {
        int32_t v = (int32_t)m->c[i];
        int32_t floor = (prev && i < prev_card && prev->c[i] == 0) ? 0 : 1;
        if (v < floor) v = floor;
        m->c[i] = (uint32_t)v; n += (uint32_t)v;
    }
    m->n = n;
    while (m->n >= CBCG_RESCALE) {                             /* update_model's halve-and-increment, src/stream_model.c:38-49 */
        m->n = 0;
        for (uint32_t i = 0; i < m->card; i++) { m->c[i] = (m->c[i] >> 1) + 1; m->n += m->c[i]; }
    }
}
/* FLAG: clamp, then scale to the target total instead of halving (cbcg_flag_target, cbcg_format.h). */
static uint32_t finish_flag(model *m, uint32_t target) {
    uint64_t n = 0;
    for (uint32_t i = 0; i < m->card; i++) { int32_t v = (int32_t)m->c[i]; if (v < 1) v = 1; m->c[i] = (uint32_t)v; n += (uint32_t)v; }
    if (n > target) {
        const uint64_t a = target - 65536u;
        uint64_t s = 0;
        for (uint32_t i = 0; i < m->card; i++) { uint64_t c = (uint64_t)m->c[i] * a / n; if (c < 1) c = 1; m->c[i] = (uint32_t)c; s += c; }
        n = s;
    }
    /* rule F2 (cbcg_format.h): at most CBCG_FLAG_ADAPT_MAX counts differ from 1 in a snapshot */
    uint32_t adapted = 0;
    for (uint32_t i = 0; i < m->card; i++) adapted += m->c[i] != 1u;
    if (adapted > CBCG_FLAG_ADAPT_MAX) {
        uint32_t lo = 1u, hi = 0x7fffffffu;
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo) / 2u;
            uint32_t above = 0;
            for (uint32_t i = 0; i < m->card; i++) above += m->c[i] > mid;
            if (above <= CBCG_FLAG_ADAPT_MAX) hi = mid; else lo = mid + 1u;
        }
        n = 0; adapted = 0;
        for (uint32_t i = 0; i < m->card; i++) { if (m->c[i] <= lo) m->c[i] = 1u; n += m->c[i]; adapted += m->c[i] != 1u; }
    }
    m->n = (uint32_t)n;
    return adapted;
}
static void merge_finish(models *acc, const models *prev, uint32_t flag_target) {
    for (int i = 0; i < 4; i++) { finish_model(&acc->rlength[i], &prev->rlength[i], 255); finish_model(&acc->pos_alpha[i], &prev->pos_alpha[i], 256);
                                  finish_model(&acc->match[i], &prev->match[i], 2); }
    for (int i = 0; i < 6; i++) finish_model(&acc->chars[i], &prev->chars[i], 5);
    finish_model(&acc->same_ref, &prev->same_ref, 2);
    acc->flag_adapted = finish_flag(&acc->flag, flag_target);
    finish_model(&acc->snps, &prev->snps, acc->L); finish_model(&acc->indels, &prev->indels, acc->L);
    for (uint32_t ctx = 0; ctx < CBCG_VAR_CONTEXTS; ctx++) if (acc->var[ctx].c) finish_model(&acc->var[ctx], NULL, 0);
    finish_model(&acc->pos.m, NULL, 0);
    /* the snapshot must stand alone: pull in the rows it still shares with its predecessor */
    for (uint32_t ctx = 0; ctx < CBCG_VAR_CONTEXTS; ctx++) if (!acc->var[ctx].c && prev->var[ctx].c) (void)model_of(acc, CBCG_S_VAR, ctx);
    acc->base = NULL;
}

static model *model_of(models *M, uint32_t stream, uint32_t ctx) {
    switch (stream) {
        case CBCG_S_CODEBOOK:  return ctx < 4 ? &M->codebook[ctx] : NULL;
        case CBCG_S_SAME_REF:  return ctx == 0 ? &M->same_ref : NULL;
        case CBCG_S_RNAME:     return ctx < 256 ? &M->rname[ctx] : NULL;
        case CBCG_S_RLENGTH:   return ctx < 4 ? &M->rlength[ctx] : NULL;
        case CBCG_S_POS:       return &M->pos.m;
        case CBCG_S_POS_ALPHA: return ctx < 4 ? &M->pos_alpha[ctx] : NULL;
        case CBCG_S_FLAG:      return &M->flag;
        case CBCG_S_MATCH:     return ctx < 4 ? &M->match[ctx] : NULL;
        case CBCG_S_SNPS:      return &M->snps;
        case CBCG_S_INDELS:    return &M->indels;
        case CBCG_S_CHARS:     return ctx < 6 ? &M->chars[ctx] : NULL;
        case CBCG_S_VAR:
            if (ctx >= CBCG_VAR_CONTEXTS) return NULL;
            if (!M->var[ctx].c) {
                if (M->base && M->base->var[ctx].c) {
                    const model *src = &M->base->var[ctx];
                    model *d = &M->var[ctx];
                    d->c = (uint32_t *)malloc(sizeof(uint32_t) * src->card);
                    memcpy(d->c, src->c, sizeof(uint32_t) * src->card);
                    d->card = src->card; d->step = src->step; d->n = src->n;
                } else model_ones(&M->var[ctx], M->L, 10);
            }
            return &M->var[ctx];
        default: return NULL;
    }
}

/* ------------------------------------------------------------------ coder front end
 * One object for the three uses of the read-level logic: trace only, encode, decode. */
typedef struct {
    models M;
    acoder ac[CBCG_N_SUB];  /* legacy stream: ac[0] codes everything; blocked containers: one coder per substream */
    int split;              /* 1: blocked container v4, symbols go to the substream of their model (cbcg_substream_of) */
    uint32_t sub_syms[CBCG_N_SUB];
    int mode;               /* 0 trace only, 1 encode, 2 decode */
    int flag_bound;         /* blocked containers: rule F1 (cbcg_format.h) */
    cbco_buf *trace;        /* optional (key, symbol) log, tracer format */
    int err;
    uint64_t n_symbols;
} coder;

/* Rule F1 (cbcg_format.h): a block adapts at most CBCG_FLAG_ADAPT_MAX distinct FLAG values; a further new value has
 * just been coded with its count of 1 and leaves the model as it was. Returns 1 when the update is to be skipped. */
static int flag_saturated(coder *c, const model *m, uint32_t x) {
    if (m->c[x] != 1u) return 0;                              /* already adapted */
    if (c->flag_bound && c->M.flag_adapted >= CBCG_FLAG_ADAPT_MAX) return 1;
    c->M.flag_adapted++;
    return 0;
}
/* send_value_to_as + update_model (src/stream_model.c:53-76,31-51) */
static void put_sym(coder *c, uint32_t stream, uint32_t ctx, uint32_t x) {
    if (c->err) return;
    model *m = model_of(&c->M, stream, ctx);
    if (!m || x >= m->card) { c->err = -2; return; }           /* reference: assert :62 */
    if (c->trace) { uint32_t rec[2] = { CBCG_SYM_KEY(stream, ctx), x }; buf_put(c->trace, rec, 8); }
    c->n_symbols++;
    if (c->mode == 1) {
        uint32_t lo = 0;
        for (uint32_t i = 0; i < x; i++) lo += m->c[i];
        const uint32_t sub = c->split ? cbcg_substream_of(stream) : 0u;
        c->sub_syms[sub]++;
        if (ac_encode(&c->ac[sub], lo, lo + m->c[x], m->n)) { c->err = -3; return; }   /* assert :71 */
    }
    if (stream == CBCG_S_FLAG && flag_saturated(c, m, x)) return;
    model_update(m, x);
}
/* read_value_from_as + update_model (src/stream_model.c:78-117) */
static uint32_t get_sym(coder *c, uint32_t stream, uint32_t ctx) {
    if (c->err) return 0;
    model *m = model_of(&c->M, stream, ctx);
    if (!m) { c->err = -2; return 0; }
    acoder *ac = &c->ac[c->split ? cbcg_substream_of(stream) : 0u];
    uint32_t target = ac_target(ac, m->n);
    uint32_t x = 0, cum = 0;
    while (cum <= target) {
        if (x >= m->card) { c->err = -4; return 0; }           /* corrupt stream */
        cum += m->c[x++];
    }
    x--;
    uint32_t lo = cum - m->c[x];
    ac_decode(ac, lo, cum, m->n);
    if (c->trace) { uint32_t rec[2] = { CBCG_SYM_KEY(stream, ctx), x }; buf_put(c->trace, rec, 8); }
    c->n_symbols++;
    if (stream == CBCG_S_FLAG && flag_saturated(c, m, x)) return x;
    model_update(m, x);
    return x;
}

/* compress_int / decompress_int: src/qv_codebook.c:14-95 */
__attribute__((unused)) static void put_int(coder *c, uint32_t v) {
    for (int k = 0; k < 4; k++) put_sym(c, CBCG_S_CODEBOOK, (uint32_t)k, (v >> (24 - 8 * k)) & 0xffu);
}
static uint32_t get_int(coder *c) {
    uint32_t v = 0;
    for (int k = 0; k < 4; k++) v |= get_sym(c, CBCG_S_CODEBOOK, (uint32_t)k) << (24 - 8 * k);
    return v;
}

/* compress_pos / compress_pos_alpha: src/read_compression.c:75-159 */
static void put_pos(coder *c, uint32_t x) {
    int slot = pos_find(&c->M.pos, x);
    if (slot >= 0) { put_sym(c, CBCG_S_POS, 0, (uint32_t)slot); return; }
    put_sym(c, CBCG_S_POS, 0, 0);
    for (int k = 0; k < 4; k++) put_sym(c, CBCG_S_POS_ALPHA, (uint32_t)k, (x >> (24 - 8 * k)) & 0xffu);
    uint32_t s = pos_append(&c->M.pos, x);
    model_update(&c->M.pos.m, s);                       /* :153, no coder step */
}
/* decompress_pos / decompress_pos_alpha: src/read_decompression.c:144-228 */
static uint32_t get_pos(coder *c) {
    uint32_t slot = get_sym(c, CBCG_S_POS, 0);
    if (c->err) return 0;
    if (slot != 0) return c->M.pos.alpha[slot];
    uint32_t x = 0;
    for (int k = 0; k < 4; k++) x |= get_sym(c, CBCG_S_POS_ALPHA, (uint32_t)k) << (24 - 8 * k);
    uint32_t s = pos_append(&c->M.pos, x);
    model_update(&c->M.pos.m, s);
    return x;
}

/* ------------------------------------------------------------------ SNP-site memory
 * snpInRef[] (include/read_compression.h:28): one byte per reference position of the
 * current chromosome, set at every SNP site seen so far. Kept with an undo list so a
 * block-local copy can be cleared cheaply. */
typedef struct { uint8_t *mark; uint64_t cap; uint64_t *touched; uint64_t nt, tcap; } snpmem;
static void snp_reset(snpmem *s, uint64_t need) {
    if (need > s->cap) { free(s->mark); s->mark = (uint8_t *)calloc(need, 1); s->cap = need; s->nt = 0; return; }
    for (uint64_t i = 0; i < s->nt; i++) s->mark[s->touched[i]] = 0;
    s->nt = 0;
}
static void snp_set(snpmem *s, uint64_t i) {
    if (i >= s->cap || s->mark[i]) return;
    s->mark[i] = 1;
    if (s->nt == s->tcap) { s->tcap = s->tcap ? s->tcap * 2 : 1024; s->touched = (uint64_t *)realloc(s->touched, 8 * s->tcap); }
    s->touched[s->nt++] = i;
}
static void snp_free(snpmem *s) { free(s->mark); free(s->touched); memset(s, 0, sizeof *s); }
/* compute_delta_to_first_snp: src/read_compression.c:703-718 (cumsumP == pos) */
static uint32_t snp_delta(const snpmem *s, uint32_t pos, uint32_t prev, uint32_t len) {
    for (uint32_t j = 0; j + prev < len; j++) {
        uint64_t i = (uint64_t)pos - 1 + j + prev;
        if (i < s->cap && s->mark[i]) return j;
    }
    return len + 2;
}

/* ------------------------------------------------------------------ edit extraction
 * compress_edits (:265-606) and the resumable MD walker add_snps_to_array (:613-701),
 * src/read_compression.c. */
static uint32_t num_digits(uint32_t x) {     /* compute_num_digits :720-743 */
    uint32_t d = 1;
    while (x >= 10 && d < 9) { x /= 10; d++; }
    return d;
}
static uint32_t md_atoi(const uint8_t *p, const uint8_t *end) {
    uint32_t v = 0;
    while (p < end && *p >= '0' && *p <= '9') v = v * 10 + (uint32_t)(*p++ - '0');
    return v;
}
typedef struct { const uint8_t *md, *end; uint32_t ptr, cum; int done; } mdwalk;
typedef struct { uint32_t pos; uint8_t refb, target; } snp_t;

static int md_ch(const mdwalk *w, uint32_t off) { return (w->md + off < w->end) ? w->md[off] : 0; }

/* Returns non-zero while SNPs may remain (the caller keeps calling), 0 when MD is used up. */
static int md_walk(mdwalk *w, snp_t *snps, uint32_t *n_snps, uint32_t insertion_pos,
                   const uint8_t *read, uint32_t read_len) {
    while (md_ch(w, w->ptr) != 0) {
        /* look ahead: matches up to the next mismatch, across deletions (:626-649) */
        uint32_t pos = md_atoi(w->md + w->ptr, w->end), temp = pos;
        uint32_t o = w->ptr + num_digits(pos);
        int ch = md_ch(w, o); o++;
        int hit_end = 0;
        while (ch == '^') {
            while (md_ch(w, o) != 0 && !isdigit(md_ch(w, o))) o++;
            uint32_t v = md_atoi(w->md + o, w->end);
            temp += v; o += num_digits(v);
            ch = md_ch(w, o); o++;
            if (ch == 0) { hit_end = 1; break; }
        }
        if (hit_end) break;
        if (w->cum + temp >= insertion_pos) { w->cum++; return 1; }       /* :656-659 */
        /* consume (:661-682) */
        w->ptr += num_digits(pos);
        ch = md_ch(w, w->ptr); w->ptr++;
        while (ch == '^') {
            while (md_ch(w, w->ptr) != 0 && !isdigit(md_ch(w, w->ptr))) w->ptr++;
            uint32_t v = md_atoi(w->md + w->ptr, w->end);
            pos += v; w->ptr += num_digits(v);
            ch = md_ch(w, w->ptr); w->ptr++;
        }
        if (ch == 0) break;
        w->cum += pos;
        snps[*n_snps].pos = pos;
        snps[*n_snps].refb = (uint8_t)base_code(ch);
        snps[*n_snps].target = (uint8_t)base_code(w->cum < read_len ? read[w->cum] : 0);
        (*n_snps)++;
        w->cum++;
        if (md_ch(w, w->ptr) == 0) break;
    }
    w->ptr = 0; w->cum = 0; w->done = 1;
    return 0;
}

/* One read. Returns 0, or <0 when the read is outside what the reference can code (-2: its edits do not fit in
 * edits_cap entries). */
static int extract_read(const uint8_t *read, uint32_t len, const uint8_t *cigar, uint32_t cigar_len,
                        const uint8_t *md, uint32_t md_len, const uint8_t *ref, uint64_t ref_len,
                        uint32_t pos, cbcg_read_rec *rec, uint16_t *edits, uint64_t edits_cap, uint32_t *n_edits) {
    *n_edits = 0;
    rec->match = 0; rec->n_snps = rec->n_dels = rec->n_ins = 0;
    if (pos == 0 || len == 0 || len > CBCG_MAX_READ_LEN) return -10;
    /* perfect-match test, independent of CIGAR/MD (:291-296) */
    int matches = ((uint64_t)pos - 1 + len <= ref_len);
    for (uint32_t i = 0; matches && i < len; i++) if (read[i] != ref[pos - 1 + i]) matches = 0;
    if (matches) { rec->match = 1; return 0; }

    static __thread uint32_t dels[1024];
    static __thread struct { uint32_t pos; uint8_t target; } ins[1024];
    static __thread snp_t snps[1024];
    uint32_t n_ins = 0, n_dels = 0, n_snps = 0;
    uint32_t M = 0, prev_i = 0, prev_d = 0;
    int last_snp = 1, first = 1;
    mdwalk w = { md, md + md_len, 0, 0, 0 };

    uint32_t i = 0;
    while (i < cigar_len) {
        uint32_t num = 0, j = i;
        while (j < cigar_len && cigar[j] >= '0' && cigar[j] <= '9') num = num * 10 + (uint32_t)(cigar[j++] - '0');
        if (j >= cigar_len) return -11;
        int op = cigar[j];
        switch (op) {
            case 'M': case '=': case 'X':        /* reference handles only 'M' (:312) */
                M += num; break;
            case 'I':                            /* :321-337 */
                for (uint32_t k = 0; k < num; k++) {
                    if (n_ins >= 1000) return -12;
                    if (last_snp) last_snp = md_walk(&w, snps, &n_snps, M + n_ins, read, len);
                    ins[n_ins].pos = M - prev_i;
                    ins[n_ins].target = (uint8_t)base_code(M + n_ins < len ? read[M + n_ins] : 0);
                    prev_i = M; n_ins++;
                }
                break;
            case 'D':                            /* :340-352 */
                for (uint32_t k = 0; k < num; k++) {
                    if (n_dels >= 1000) return -12;
                    dels[n_dels++] = M - prev_d; prev_d = M;
                }
                break;
            case 'S':
                if (first) {                     /* leading clip (:358-468): bases coded as insertions at 0 */
                    for (uint32_t k = 0; k < num; k++) {
                        if (n_ins >= 1000) return -12;
                        if (last_snp) last_snp = md_walk(&w, snps, &n_snps, n_ins, read, len);
                        ins[n_ins].pos = 0;
                        ins[n_ins].target = (uint8_t)base_code(k < len ? read[k] : 0);
                        n_ins++;
                    }
                } else {                         /* trailing clip (:469-479) */
                    for (uint32_t k = 0; k < num; k++) {
                        if (n_ins >= 1000) return -12;
                        ins[n_ins].pos = M - prev_i;
                        ins[n_ins].target = (uint8_t)base_code(M + n_ins < len ? read[M + n_ins] : 0);
                        prev_i = M; n_ins++;
                    }
                }
                break;
            case 'H': case 'P': break;           /* no effect on SEQ */
            default: return -13;                 /* '*', 'N', junk: the reference cannot code these */
        }
        first = 0;
        i = j + 1;
    }
    if (last_snp) md_walk(&w, snps, &n_snps, len + 1, read, len);       /* :551-552 */

    if (n_snps > 255 || n_dels > 255 || n_ins > 255) return -14;
    /* the reference span the decoder rebuilds from (rebuild_read below) must lie inside the chromosome; K1 refuses the
       same reads. Insertions and clips may carry SEQ past the chromosome's end. */
    if (n_ins > len || (uint64_t)pos - 1 + (len - n_ins) + n_dels > ref_len) return -15;
    if ((uint64_t)n_dels + n_snps + n_ins > edits_cap) return -2;
    rec->n_snps = (uint8_t)n_snps; rec->n_dels = (uint8_t)n_dels; rec->n_ins = (uint8_t)n_ins;
    uint32_t e = 0;
    for (uint32_t k = 0; k < n_dels; k++) { if (dels[k] > 255) return -14; edits[e++] = CBCG_EDIT(dels[k], 0, 0); }
    for (uint32_t k = 0; k < n_snps; k++) { if (snps[k].pos > 255) return -14; edits[e++] = CBCG_EDIT(snps[k].pos, snps[k].target, snps[k].refb); }
    for (uint32_t k = 0; k < n_ins; k++) { if (ins[k].pos > 255) return -14; edits[e++] = CBCG_EDIT(ins[k].pos, ins[k].target, CBCG_BP_O); }
    *n_edits = e;
    return 0;
}

int64_t cbco_extract(const cbco_batch *b, const cbco_genome *g, cbcg_read_rec *recs,
                     uint16_t *edits, uint64_t edits_cap) {
    uint64_t total = 0;
    for (uint64_t r = 0; r < b->n_reads; r++) {
        uint32_t chr = b->chr[r];
        if (chr >= g->n_chr) return -1;
        uint32_t len = b->seq_len[r];
        cbcg_read_rec *rec = &recs[r];
        rec->pos = b->pos[r]; rec->flag = b->flag[r]; rec->len = (uint16_t)len; rec->edit_off = (uint32_t)total;
        uint32_t ne = 0;
        int rc = extract_read(b->seq + b->seq_off[r], len,
                              b->cigar + b->cigar_off[r], (uint32_t)(b->cigar_off[r + 1] - b->cigar_off[r]),
                              b->md + b->md_off[r], (uint32_t)(b->md_off[r + 1] - b->md_off[r]),
                              g->bases[chr], g->len[chr], b->pos[r], rec, edits + total, edits_cap - total, &ne);
        if (rc) return rc;
        total += ne;
    }
    return (int64_t)total;
}

/* ------------------------------------------------------------------ reconstruction
 * reconstruct_read (src/read_decompression.c:339-529) followed by print_line
 * (src/compression.c:16-40). For reverse reads the reference builds the reverse
 * complement and print_line reverses it again, so the emitted line is the forward
 * construction for either strand. */
static int rebuild_read(const cbcg_read_rec *rec, const uint16_t *e, const uint8_t *ref, uint64_t ref_len, uint8_t *out) {
    uint32_t len = rec->len, pos = rec->pos;
    if (rec->match) {
        if ((uint64_t)pos - 1 + len > ref_len) return -1;
        memcpy(out, ref + pos - 1, len);                         /* :383-384 */
        return 0;
    }
    uint8_t tmp[1024];
    uint32_t nd = rec->n_dels, ns = rec->n_snps, ni = rec->n_ins;
    if (ni > len) return -1;
    uint32_t aligned = len - ni, cur = 0;
    if ((uint64_t)pos - 1 + aligned + nd > ref_len) return -1;
    for (uint32_t k = 0; k < nd; k++) {                          /* :418-430 */
        uint32_t d = CBCG_EDIT_DELTA(e[k]);
        for (uint32_t t = 0; t < d && cur < aligned; t++) { tmp[cur] = ref[pos + cur - 1 + k]; cur++; }
    }
    for (; cur < aligned; cur++) tmp[cur] = ref[pos + cur - 1 + nd];   /* :434-437 */
    cur = 0;
    for (uint32_t k = 0; k < ns; k++) {                          /* :442-458 */
        uint32_t p = CBCG_EDIT_DELTA(e[nd + k]);
        if (cur + p >= aligned) return -1;
        tmp[cur + p] = (uint8_t)base_char((int)CBCG_EDIT_TARGET(e[nd + k]));
        cur += p + 1;
    }
    uint32_t o = 0; cur = 0;
    for (uint32_t k = 0; k < ni; k++) {                          /* :467-483 */
        uint32_t p = CBCG_EDIT_DELTA(e[nd + ns + k]);
        for (uint32_t t = 0; t < p && cur < aligned; t++) out[o++] = tmp[cur++];
        out[o++] = (uint8_t)base_char((int)CBCG_EDIT_TARGET(e[nd + ns + k]));
    }
    while (cur < aligned) out[o++] = tmp[cur++];                 /* :486-487 */
    return o == len ? 0 : -1;
}

int64_t cbco_reconstruct(uint64_t n_reads, const cbcg_read_rec *recs, const uint16_t *edits,
                         const uint32_t *chr, const cbco_genome *g, uint8_t *out, uint64_t out_cap) {
    uint64_t o = 0;
    for (uint64_t r = 0; r < n_reads; r++) {
        if (chr[r] >= g->n_chr || o + recs[r].len + 1 > out_cap) return -1;
        if (rebuild_read(&recs[r], edits + recs[r].edit_off, g->bases[chr[r]], g->len[chr[r]], out + o)) return -2;
        o += recs[r].len;
        out[o++] = '\n';
    }
    return (int64_t)o;
}

/* ------------------------------------------------------------------ read-level coding
 * State that the reference keeps in statics/globals, made explicit (SURVEY.md section 7,
 * hard part 2): prevPos (src/read_compression.c:115), prevM (:167), prev_name/prevChar
 * (src/id_compression.c:41-42), snpInRef. */
typedef struct {
    coder c;
    uint32_t prev_pos, prev_m, prev_char;
    int have_name; uint32_t cur_chr;
    snpmem snp;
    cbco_buf *raw;          /* optional raw symbol list (POS as CBCG_S_POS_X) */
    int lean;               /* blocked containers: the per-read symbols that are constant by construction
                               (same_ref = 0, length bytes 1..3 = 0) are not coded */
    uint32_t fixed_len;     /* blocked containers of equal-length reads (CBCG_MODE_FIXED_LEN): length byte 0 is not
                               coded either; this is the length */
} rstate;

static void raw_sym(rstate *s, uint32_t stream, uint32_t ctx, uint32_t v) {
    if (s->raw) { uint32_t rec[2] = { CBCG_SYM_KEY(stream, ctx), v }; buf_put(s->raw, rec, 8); }
}
static void emit(rstate *s, uint32_t stream, uint32_t ctx, uint32_t v) {
    raw_sym(s, stream, ctx, v);
    put_sym(&s->c, stream, ctx, v);
}

/* compress_rname: src/id_compression.c:39-65 */
static void put_rname(rstate *s, const char *name) {
    emit(s, CBCG_S_SAME_REF, 0, 1);
    for (const char *p = name; *p; p++) { emit(s, CBCG_S_RNAME, s->prev_char, (uint8_t)*p); s->prev_char = (uint8_t)*p; }
    emit(s, CBCG_S_RNAME, s->prev_char, 0);
}

/* compress_read (:15-44) + the emission half of compress_edits (:557-600),
 * src/read_compression.c. chr_change resets prevPos (:123-124). */
static void put_read(rstate *s, const cbcg_read_rec *rec, const uint16_t *e) {
    uint32_t len = rec->len;
    if (!s->fixed_len) emit(s, CBCG_S_RLENGTH, 0, len & 0xffu); /* :29-33: bytes 1..3 are always 0 */
    if (!s->lean) for (uint32_t k = 1; k < 4; k++) emit(s, CBCG_S_RLENGTH, k, 0);
    uint32_t x = rec->pos - s->prev_pos + 1;                    /* :128 */
    raw_sym(s, CBCG_S_POS_X, 0, x);
    put_pos(&s->c, x);
    uint32_t same_pos = (x == 1);
    s->prev_pos = rec->pos;
    emit(s, CBCG_S_FLAG, 0, rec->flag);
    uint32_t strand = (rec->flag >> 4) & 1u;                    /* :57-60 */
    emit(s, CBCG_S_MATCH, (same_pos << 1) | s->prev_m, rec->match);   /* :164-188 */
    s->prev_m = rec->match;
    if (rec->match) return;
    uint32_t nd = rec->n_dels, ns = rec->n_snps, ni = rec->n_ins;
    if ((nd | ni) == 0) emit(s, CBCG_S_SNPS, 0, ns);
    else { emit(s, CBCG_S_SNPS, 0, 0); emit(s, CBCG_S_INDELS, 0, ns); emit(s, CBCG_S_INDELS, 0, nd); emit(s, CBCG_S_INDELS, 0, ni); }
    uint32_t prev = 0;
    for (uint32_t k = 0; k < nd; k++) { uint32_t d = CBCG_EDIT_DELTA(e[k]); emit(s, CBCG_S_VAR, (prev << 1) | strand, d); prev += d; }
    prev = 0;
    for (uint32_t k = 0; k < ns; k++) {
        uint16_t ed = e[nd + k];
        uint32_t delta = snp_delta(&s->snp, rec->pos, prev, len);
        emit(s, CBCG_S_VAR, ((((delta << CBCG_BITS_DELTA) + prev) << 1) | strand), CBCG_EDIT_DELTA(ed));
        prev += CBCG_EDIT_DELTA(ed) + 1;
        snp_set(&s->snp, (uint64_t)rec->pos + prev - 2);        /* :589 */
        emit(s, CBCG_S_CHARS, CBCG_EDIT_REFB(ed), CBCG_EDIT_TARGET(ed));
    }
    prev = 0;
    for (uint32_t k = 0; k < ni; k++) {
        uint16_t ed = e[nd + ns + k];
        emit(s, CBCG_S_VAR, (prev << 1) | strand, CBCG_EDIT_DELTA(ed)); prev += CBCG_EDIT_DELTA(ed);
        emit(s, CBCG_S_CHARS, CBCG_BP_O, CBCG_EDIT_TARGET(ed));
    }
}

/* decompress_read (:59-86) + the decoding half of reconstruct_read (:339-458,:462-511),
 * src/read_decompression.c. Fills rec/edits; needs the reference for the chars context. */
static void get_read(rstate *s, cbcg_read_rec *rec, uint16_t *e, uint32_t *n_edits,
                     const uint8_t *ref, uint64_t ref_len) {
    coder *c = &s->c;
    uint32_t len = s->fixed_len ? s->fixed_len : get_sym(c, CBCG_S_RLENGTH, 0);
    if (!s->lean) for (uint32_t k = 1; k < 4; k++) len |= get_sym(c, CBCG_S_RLENGTH, k) << (8 * k);
    uint32_t x = get_pos(c);
    uint32_t pos = s->prev_pos + x - 1;
    s->prev_pos = pos;
    uint32_t flag = get_sym(c, CBCG_S_FLAG, 0);
    uint32_t strand = (flag >> 4) & 1u;
    uint32_t match = get_sym(c, CBCG_S_MATCH, ((uint32_t)(x == 1) << 1) | s->prev_m);
    s->prev_m = match;
    rec->pos = pos; rec->flag = (uint16_t)flag; rec->len = (uint16_t)len; rec->match = (uint8_t)match;
    rec->n_snps = rec->n_dels = rec->n_ins = 0;
    *n_edits = 0;
    if (match || c->err) return;
    uint32_t ns = get_sym(c, CBCG_S_SNPS, 0), nd = 0, ni = 0;
    if (ns == 0) { ns = get_sym(c, CBCG_S_INDELS, 0); nd = get_sym(c, CBCG_S_INDELS, 0); ni = get_sym(c, CBCG_S_INDELS, 0); }
    if (c->err || ni > len || ns > 255 || nd > 255 || ni > 255) { if (!c->err) c->err = -5; return; }
    rec->n_snps = (uint8_t)ns; rec->n_dels = (uint8_t)nd; rec->n_ins = (uint8_t)ni;
    uint32_t cumdel[256];
    uint32_t prev = 0, ne = 0;
    for (uint32_t k = 0; k < nd; k++) {
        uint32_t d = get_sym(c, CBCG_S_VAR, (prev << 1) | strand); prev += d; cumdel[k] = prev;
        e[ne++] = CBCG_EDIT(d, 0, 0);
    }
    prev = 0;
    for (uint32_t k = 0; k < ns; k++) {
        uint32_t delta = snp_delta(&s->snp, pos, prev, len);
        uint32_t p = get_sym(c, CBCG_S_VAR, ((((delta << CBCG_BITS_DELTA) + prev) << 1) | strand));
        uint32_t idx = prev + p;                                /* index in the insertion-free read */
        prev += p + 1;
        snp_set(&s->snp, (uint64_t)pos + prev - 2);
        uint32_t skipped = 0;                                   /* deletions at or before idx (:426-437) */
        while (skipped < nd && cumdel[skipped] <= idx) skipped++;
        uint64_t ri = (uint64_t)pos - 1 + idx + skipped;
        uint32_t refb = (uint32_t)base_code(ri < ref_len ? ref[ri] : 0);
        uint32_t tgt = get_sym(c, CBCG_S_CHARS, refb);
        e[ne++] = CBCG_EDIT(p, tgt, refb);
        if (c->err) return;
    }
    prev = 0;
    for (uint32_t k = 0; k < ni; k++) {
        uint32_t p = get_sym(c, CBCG_S_VAR, (prev << 1) | strand); prev += p;
        uint32_t tgt = get_sym(c, CBCG_S_CHARS, CBCG_BP_O);
        e[ne++] = CBCG_EDIT(p, tgt, CBCG_BP_O);
    }
    *n_edits = ne;
}

static void rstate_init(rstate *s, uint32_t L, int mode) {
    memset(s, 0, sizeof *s);
    models_init(&s->c.M, L);
    s->c.mode = mode;
}
static void rstate_free(rstate *s) { models_free(&s->c.M); snp_free(&s->snp); }

/* ------------------------------------------------------------------ legacy single stream
 * compress() / compress_line(): src/compression.c:42-69,112-170; header writers
 * src/sam_file_allocation.c:363-404. */
static void put_header(rstate *s, uint32_t L) {
    uint32_t v[34]; v[0] = L; for (int i = 0; i < 32; i++) v[1 + i] = CBCG_WELL_DEBUG; v[33] = CBCG_LOSSLESS;
    for (int i = 0; i < 34; i++)
        for (int k = 0; k < 4; k++) emit(s, CBCG_S_CODEBOOK, (uint32_t)k, (v[i] >> (24 - 8 * k)) & 0xffu);
}

static int code_range(rstate *s, const cbco_batch *b, const cbco_genome *g, const cbcg_read_rec *recs,
                      const uint16_t *edits, uint64_t r0, uint64_t r1, int legacy) {
    for (uint64_t r = r0; r < r1; r++) {
        uint32_t chr = b->chr[r];
        int change = !s->have_name || chr != s->cur_chr;
        if (legacy) {
            if (change) put_rname(s, g->name[chr]); else emit(s, CBCG_S_SAME_REF, 0, 0);
        } else {
            if (change && r != r0) return -6;                   /* blocks never span chromosomes */
            if (!s->lean) emit(s, CBCG_S_SAME_REF, 0, 0);
        }
        if (change) {                                           /* src/compression.c:58-64 */
            s->have_name = 1; s->cur_chr = chr;
            if (legacy) s->prev_pos = 0;
            snp_reset(&s->snp, g->len[chr] + 2048);
        }
        /* single stream: the reference indexes alphaExist / alphaMap, CBCG_MAX_POS_X entries each (sam_block.h:54), by the
           POS step, so a step above CBCG_MAX_POS_X is refused, as the GPU encoder refuses it. Whether the reference itself
           survives a step of exactly CBCG_MAX_POS_X was never run against its binary. A blocked container codes any
           32-bit step through the escape and has no such limit. */
        if (legacy && recs[r].pos - s->prev_pos + 1u > CBCG_MAX_POS_X) return -16;
        put_read(s, &recs[r], edits + recs[r].edit_off);
        if (s->c.err) return s->c.err;
    }
    return 0;
}

int cbco_encode_legacy(const cbco_batch *b, const cbco_genome *g, uint32_t L, cbco_buf *out, cbco_buf *trace) {
    uint64_t cap = 16;
    for (uint64_t r = 0; r < b->n_reads; r++) cap += CBCO_EDITS_PER_READ(b->seq_len[r]);
    cbcg_read_rec *recs = (cbcg_read_rec *)malloc(sizeof(cbcg_read_rec) * (b->n_reads + 1));
    uint16_t *edits = (uint16_t *)malloc(2 * cap);
    int64_t ne = cbco_extract(b, g, recs, edits, cap);
    int rc = ne < 0 ? (int)ne : 0;
    if (!rc) {
        rstate s; rstate_init(&s, L, 1);
        s.c.trace = trace;
        ac_init_enc(&s.c.ac[0], out);
        put_header(&s, L);
        rc = code_range(&s, b, g, recs, edits, 0, b->n_reads, 1);
        if (!rc) {
            put_rname(&s, "\n");                                /* src/compression.c:152 */
            ac_flush(&s.c.ac[0]);
            rc = s.c.err;
        }
        rstate_free(&s);
    }
    free(recs); free(edits);
    return rc;
}

/* decompress() / decompress_line(): src/compression.c:71-108,173-216;
 * decompress_rname src/id_compression.c:67-94. Chromosomes are taken in FASTA order, as
 * the reference does (it reads the next FASTA record on every name change). */
int cbco_decode_legacy(const uint8_t *stream, uint64_t stream_len, const cbco_genome *g,
                       cbco_buf *seq_out, uint64_t *n_reads_out) {
    rstate s; rstate_init(&s, 1, 2);
    ac_init_dec(&s.c.ac[0], stream, stream_len);
    uint32_t L = get_int(&s.c);
    for (int i = 0; i < 32; i++) (void)get_int(&s.c);
    uint32_t lossiness = get_int(&s.c);
    int rc = 0;
    uint64_t n = 0;
    if (s.c.err || L == 0 || L > 1024 || lossiness != CBCG_LOSSLESS) rc = -20;
    else {
        /* models that depend on L are (re)built now, as alloc_read_block_t does after the header int */
        models_free(&s.c.M); models_init(&s.c.M, L);
        /* keep the codebook state? It is not used past the header. */
        int32_t chr = -1;
        uint16_t e[3 * 256 + 8];
        uint8_t line[1024 + 1];
        for (;;) {
            uint32_t change = get_sym(&s.c, CBCG_S_SAME_REF, 0);
            if (s.c.err) { rc = s.c.err; break; }
            if (change) {
                int end = 0; uint32_t ch;
                while ((ch = get_sym(&s.c, CBCG_S_RNAME, s.prev_char)) != 0) {
                    if (s.c.err) break;
                    if (ch == '\n') { end = 1; break; }
                    s.prev_char = ch;
                }
                if (s.c.err) { rc = s.c.err; break; }
                if (end) break;
                chr++;
                if ((uint32_t)chr >= g->n_chr) { rc = -21; break; }
                s.prev_pos = 0;
                snp_reset(&s.snp, g->len[chr] + 2048);
            }
            if (chr < 0) { rc = -22; break; }
            cbcg_read_rec rec; uint32_t ne = 0;
            get_read(&s, &rec, e, &ne, g->bases[chr], g->len[chr]);
            if (s.c.err) { rc = s.c.err; break; }
            rec.edit_off = 0;
            if (rec.len > 1024 || rebuild_read(&rec, e, g->bases[chr], g->len[chr], line)) { rc = -23; break; }
            line[rec.len] = '\n';
            buf_put(seq_out, line, rec.len + 1u);
            n++;
        }
    }
    if (n_reads_out) *n_reads_out = n;
    rstate_free(&s);
    return rc;
}

int cbco_symbols(const cbco_batch *b, const cbco_genome *g, const cbcg_read_rec *recs,
                 const uint16_t *edits, uint64_t r0, uint64_t r1, uint32_t L, int legacy, cbco_buf *symbols) {
    rstate s; rstate_init(&s, L, 0);
    s.raw = symbols;
    int rc = 0;
    if (legacy) put_header(&s, L);
    else if (r0 < r1) { s.prev_pos = recs[r0].pos; s.have_name = 1; s.cur_chr = b->chr[r0]; snp_reset(&s.snp, g->len[b->chr[r0]] + 2048); }
    rc = code_range(&s, b, g, recs, edits, r0, r1, legacy);
    if (!rc && legacy) put_rname(&s, "\n");
    rstate_free(&s);
    return rc;
}

/* ------------------------------------------------------------------ blocked container
 * Our design (the reference stream has no framing). Layout, little endian:
 *   header  : u32 magic, version, max_read_len, read_len, u64 n_reads, u32 n_blocks, n_chr,
 *             block_reads, gen_mode, then per chromosome u32 name_len + bytes (padded to 4)
 *   index   : n_blocks x 8 u32 { n_reads, chr, base_pos, n_symbols, n_edits, payload_bytes, gen, 0 }
 *   payload : block bitstreams back to back
 * Each block: models at the reference's initial state (gen 0), fresh coder, prevPos = base_pos
 * (= POS of its first read), prevM = 0, empty SNP-site memory; per read the reference's symbol
 * order with same_ref = 0; closed by the reference's final flush. */
typedef struct { uint32_t n_reads, chr, base_pos, n_symbols, n_edits, payload_bytes, gen, rsv; uint32_t sub_bytes[CBCG_N_SUB]; } blk_index;

/* Index entries are delta-coded LEB128 varints (DESIGN.md, "Container"). */
static void put_varint(cbco_buf *b, uint64_t v) {
    do { uint8_t c = (uint8_t)(v & 0x7f); v >>= 7; if (v) c |= 0x80; buf_put(b, &c, 1); } while (v);
}
static uint64_t zigzag(int64_t v) { return ((uint64_t)v << 1) ^ (uint64_t)(v >> 63); }
static int64_t unzigzag(uint64_t v) { return (int64_t)(v >> 1) ^ -(int64_t)(v & 1); }
static int get_varint(const uint8_t *p, uint64_t len, uint64_t *o, uint64_t *v) {
    uint64_t r = 0; int sh = 0;
    for (;;) {
        if (*o >= len || sh > 63) return -1;
        uint8_t c = p[(*o)++];
        r |= (uint64_t)(c & 0x7f) << sh; sh += 7;
        if (!(c & 0x80)) break;
    }
    *v = r; return 0;
}
typedef struct { int64_t n_reads, chr, gen, base, d1, edits, sub[CBCG_N_SUB]; } idx_state;
static void index_put(cbco_buf *b, idx_state *st, const blk_index *e, uint32_t n_sub) {
    int chr_ch = (int64_t)e->chr != st->chr, gen_ch = (int64_t)e->gen != st->gen;
    put_varint(b, (zigzag((int64_t)e->n_reads - st->n_reads) << 2) | (chr_ch ? 2u : 0u) | (gen_ch ? 1u : 0u));
    if (chr_ch) { put_varint(b, e->chr); st->base = 0; st->d1 = 0; }
    if (gen_ch) put_varint(b, (uint64_t)((int64_t)e->gen - st->gen - 1));
    int64_t d1 = (int64_t)e->base_pos - st->base;
    put_varint(b, zigzag(d1 - st->d1));
    put_varint(b, zigzag((int64_t)e->n_edits - st->edits));
    for (uint32_t k = 0; k < n_sub; k++) { put_varint(b, zigzag((int64_t)e->sub_bytes[k] - st->sub[k])); st->sub[k] = e->sub_bytes[k]; }
    st->n_reads = e->n_reads; st->chr = e->chr; st->gen = e->gen; st->base = e->base_pos; st->d1 = d1;
    st->edits = e->n_edits;
}
static int index_get(const uint8_t *p, uint64_t len, uint64_t *o, idx_state *st, blk_index *e, uint32_t mode) {
    uint64_t v;
    if (get_varint(p, len, o, &v)) return -1;
    st->n_reads += unzigzag(v >> 2);
    if (v & 2) { uint64_t c; if (get_varint(p, len, o, &c)) return -1; st->chr = (int64_t)c; st->base = 0; st->d1 = 0; }
    if (v & 1) { uint64_t gi; if (get_varint(p, len, o, &gi)) return -1; st->gen += (int64_t)gi + 1; }
    if (get_varint(p, len, o, &v)) return -1;
    st->d1 += unzigzag(v); st->base += st->d1;
    if (get_varint(p, len, o, &v)) return -1;
    st->edits += unzigzag(v);
    int64_t total = 0;
    const uint32_t n_sub = CBCG_BLOCK_NSUB(mode, st->gen);
    for (uint32_t k = 0; k < n_sub; k++) {
        if (get_varint(p, len, o, &v)) return -1;
        st->sub[k] += unzigzag(v);
        if (st->sub[k] < 0 || st->sub[k] > 0x3fffffffll) return -1;
        total += st->sub[k];
    }
    if (st->n_reads < 0 || st->n_reads > 0xffffffffll || st->chr < 0 || st->gen < 0 || st->gen > 255 || st->base < 0 || st->base > 0xffffffffll ||
        st->edits < 0 || st->edits > 0xffffffffll || total > 0xffffffffll) return -1;
    memset(e, 0, sizeof *e);
    e->n_reads = (uint32_t)st->n_reads; e->chr = (uint32_t)st->chr; e->gen = (uint32_t)st->gen; e->base_pos = (uint32_t)st->base;
    e->n_edits = (uint32_t)st->edits; e->payload_bytes = (uint32_t)total;
    for (uint32_t k = 0; k < n_sub; k++) e->sub_bytes[k] = (uint32_t)st->sub[k];
    return 0;
}

static void rstate_init_from(rstate *s, const models *snap, int mode) {
    memset(s, 0, sizeof *s);
    models_clone(&s->c.M, snap);
    s->c.mode = mode;
    s->c.flag_bound = 1;                                       /* every block of a blocked container */
}

/* Blocks: generation i < n_sched has sched_count[i] blocks of sched_reads[i] reads, the last generation
 * takes the rest in blocks of block_reads reads; a chromosome change always ends a block. n_sched == 0:
 * every block starts from the reference's initial state (gen_mode 0). */
static int encode_cut(const cbco_batch *b, const cbco_genome *g, uint32_t L, uint32_t block_reads, uint32_t n_sched,
                      const uint32_t *sched_count, const uint32_t *sched_reads, const blk_index *given, uint64_t n_given,
                      uint32_t gen_mode, cbco_buf *out);

int cbco_encode_scheduled(const cbco_batch *b, const cbco_genome *g, uint32_t L, uint32_t block_reads,
                          uint32_t n_sched, const uint32_t *sched_count, const uint32_t *sched_reads, cbco_buf *out) {
    return encode_cut(b, g, L, block_reads & 0x7fffffffu, n_sched, sched_count, sched_reads, NULL, 0, (n_sched ? 1u : 0u) | ((block_reads & 0x80000000u) ? CBCG_MODE_SPLIT4 : 0u), out);   /* experiments: bit 31 of block_reads asks for four substreams */
}

/* The batch coded with the block cut of an existing container (per-block read counts and generations taken from its
 * index; header block size and mode word too): the check for cuts the encoder chose itself (the pipelined cbcg_encode
 * sizes last-generation blocks by their place in the batch). */
int cbco_encode_like(const uint8_t *p, uint64_t len, const cbco_batch *b, const cbco_genome *g, cbco_buf *out) {
    if (len < 40) return -40;
    uint32_t h[10]; memcpy(h, p, 40);
    if (h[0] != CBCG_MAGIC || h[1] != CBCG_VERSION) return -41;
    uint32_t nb = h[6], n_chr = h[7];
    uint64_t o = 40;
    for (uint32_t c = 0; c < n_chr; c++) {
        if (o + 4 > len) return -43;
        uint32_t nl; memcpy(&nl, p + o, 4); o += 4 + nl + ((4 - (nl & 3)) & 3);
    }
    if (o + 4 > len) return -43;
    uint32_t ix_bytes; memcpy(&ix_bytes, p + o, 4); o += 4;
    if (o + ix_bytes > len) return -43;
    blk_index *idx = (blk_index *)calloc((size_t)nb + 1, sizeof(blk_index));
    idx_state st = { h[8], 0, 0, 0, 0, 0, { 0, 0, 0, 0 } };
    uint64_t io = o;
    for (uint32_t k = 0; k < nb; k++) if (index_get(p, o + ix_bytes, &io, &st, &idx[k], h[9])) { free(idx); return -43; }
    int rc = encode_cut(b, g, h[3], h[8], (h[9] & CBCG_MODE_GEN_MASK) ? 1u : 0u, NULL, NULL, idx, nb, h[9] & (CBCG_MODE_GEN_MASK | CBCG_MODE_LAYOUT_MASK), out);
    free(idx);
    return rc;
}

static int encode_cut(const cbco_batch *b, const cbco_genome *g, uint32_t L, uint32_t block_reads, uint32_t n_sched,
                      const uint32_t *sched_count, const uint32_t *sched_reads, const blk_index *given, uint64_t n_given,
                      uint32_t gen_mode, cbco_buf *out) {
    if (block_reads == 0) return -30;
    uint64_t cap = 16;
    for (uint64_t r = 0; r < b->n_reads; r++) cap += CBCO_EDITS_PER_READ(b->seq_len[r]);
    cbcg_read_rec *recs = (cbcg_read_rec *)malloc(sizeof(cbcg_read_rec) * (b->n_reads + 1));
    uint16_t *edits = (uint16_t *)malloc(2 * cap);
    int64_t ne = cbco_extract(b, g, recs, edits, cap);
    if (ne < 0) { free(recs); free(edits); return (int)ne; }
    /* cut blocks */
    uint64_t nb = 0, bcap = 1024;
    blk_index *idx = (blk_index *)calloc(bcap, sizeof(blk_index));
    uint64_t *first = (uint64_t *)calloc(bcap + 1, sizeof(uint64_t));
    uint32_t gen = 0, left_in_gen = (n_sched && !given) ? sched_count[0] : 0;
    while (!given && gen < n_sched && left_in_gen == 0) { gen++; left_in_gen = gen < n_sched ? sched_count[gen] : 0; }
    for (uint64_t r = 0; r < b->n_reads;) {
        uint32_t want = given ? 0u : (gen < n_sched ? sched_reads[gen] : block_reads);
        if (given) {                                           /* the cut of an existing container */
            if (nb >= n_given || given[nb].n_reads == 0) { free(idx); free(first); free(recs); free(edits); return -48; }
            want = given[nb].n_reads; gen = given[nb].gen;
        }
        if (want == 0) want = 1;
        uint64_t e = r + 1;
        while (e < b->n_reads && e - r < want && b->chr[e] == b->chr[r]) e++;
        if (given && e - r != want) { free(idx); free(first); free(recs); free(edits); return -48; }
        if (nb + 1 >= bcap) { bcap *= 2; idx = (blk_index *)realloc(idx, bcap * sizeof(blk_index)); first = (uint64_t *)realloc(first, (bcap + 1) * 8); }
        first[nb] = r;
        memset(&idx[nb], 0, sizeof(blk_index));
        idx[nb].n_reads = (uint32_t)(e - r); idx[nb].chr = b->chr[r]; idx[nb].base_pos = recs[r].pos; idx[nb].gen = gen;
        nb++; r = e;
        if (given) continue;
        if (gen < n_sched && --left_in_gen == 0) { gen++; while (gen < n_sched && sched_count[gen] == 0) gen++; left_in_gen = gen < n_sched ? sched_count[gen] : 0; }
    }
    first[nb] = b->n_reads;
    const uint32_t last_gen = nb ? idx[nb - 1].gen : 0;
    uint32_t max_block = 0;
    for (uint64_t k = 0; k < nb; k++) if (idx[k].n_reads > max_block) max_block = idx[k].n_reads;
    const uint32_t flag_target = cbcg_flag_target(max_block);
    uint32_t fixed_len = b->n_reads ? L : 0;                   /* every read exactly L bases: CBCG_MODE_FIXED_LEN */
    for (uint64_t r = 0; r < b->n_reads; r++) if (b->seq_len[r] != L) { fixed_len = 0; break; }
    cbco_buf payload = {0};
    int rc = 0;
    models *prev = (models *)malloc(sizeof(models)), *acc = NULL;
    models_init(prev, L);
    uint32_t cur_gen = 0;
    for (uint64_t k = 0; k < nb && !rc; k++) {
        if (idx[k].gen != cur_gen) {                           /* generation boundary: the merged state becomes the snapshot */
            if (acc) { merge_finish(acc, prev, flag_target); models_free(prev); free(prev); prev = acc; acc = NULL; }
            cur_gen = idx[k].gen;
        }
        if (!acc && idx[k].gen != last_gen) { acc = (models *)malloc(sizeof(models)); models_clone(acc, prev); }
        rstate s; rstate_init_from(&s, prev, 1);
        s.lean = 1; s.fixed_len = fixed_len;
        uint64_t start = payload.size;
        cbco_buf sub[CBCG_N_SUB]; memset(sub, 0, sizeof sub);
        const uint32_t n_sub = CBCG_BLOCK_NSUB(gen_mode, idx[k].gen);
        s.c.split = n_sub > 1u;
        for (uint32_t q = 0; q < n_sub; q++) ac_init_enc(&s.c.ac[q], &sub[q]);
        s.prev_pos = idx[k].base_pos; s.have_name = 1; s.cur_chr = idx[k].chr;
        snp_reset(&s.snp, g->len[idx[k].chr] + 2048);
        rc = code_range(&s, b, g, recs, edits, first[k], first[k + 1], 0);
        for (uint32_t q = 0; q < n_sub; q++) {                   /* A | B | C | D, each with its own short tail; nothing coded: nothing stored */
            const int any = n_sub == 1u || s.c.sub_syms[q];         /* a single-stream block always closes its stream */
            if (!rc && any) ac_flush_short(&s.c.ac[q]);
            idx[k].sub_bytes[q] = (!rc && any) ? (uint32_t)sub[q].size : 0u;
            if (idx[k].sub_bytes[q]) buf_put(&payload, sub[q].data, sub[q].size);
            cbco_buf_free(&sub[q]);
        }
        if (!rc) rc = s.c.err;
        idx[k].n_symbols = (uint32_t)s.c.n_symbols;
        uint64_t e_lo = recs[first[k]].edit_off;
        uint64_t e_hi = (first[k + 1] < b->n_reads) ? recs[first[k + 1]].edit_off : (uint64_t)ne;
        idx[k].n_edits = (uint32_t)(e_hi - e_lo);
        idx[k].payload_bytes = (uint32_t)(payload.size - start);
        if (acc && !rc) merge_block(acc, &s.c.M, prev);
        rstate_free(&s);
    }
    if (acc) { models_free(acc); free(acc); }
    models_free(prev); free(prev);
    if (!rc) {
        uint32_t max_len = 0;
        for (uint64_t r = 0; r < b->n_reads; r++) if (b->seq_len[r] > max_len) max_len = b->seq_len[r];
        buf_put_u32(out, CBCG_MAGIC); buf_put_u32(out, CBCG_VERSION); buf_put_u32(out, max_len); buf_put_u32(out, L);
        buf_put_u64(out, b->n_reads); buf_put_u32(out, (uint32_t)nb); buf_put_u32(out, g->n_chr);
        buf_put_u32(out, block_reads); buf_put_u32(out, gen_mode | (fixed_len ? CBCG_MODE_FIXED_LEN : 0u));   /* gen_mode: generations | CBCG_MODE_SPLIT4 */
        for (uint32_t c = 0; c < g->n_chr; c++) {
            uint32_t nl = (uint32_t)strlen(g->name[c]), pad = (4 - (nl & 3)) & 3; uint32_t z = 0;
            buf_put_u32(out, nl); buf_put(out, g->name[c], nl); buf_put(out, &z, pad);
        }
        cbco_buf ix = {0};
        idx_state st = { block_reads, 0, 0, 0, 0, 0, { 0, 0, 0, 0 } };
        for (uint64_t k = 0; k < nb; k++) index_put(&ix, &st, &idx[k], CBCG_BLOCK_NSUB(gen_mode, idx[k].gen));
        buf_put_u32(out, (uint32_t)ix.size);
        buf_put(out, ix.data, ix.size);
        cbco_buf_free(&ix);
        buf_put(out, payload.data, payload.size);
    }
    cbco_buf_free(&payload);
    free(idx); free(first); free(recs); free(edits);
    return rc;
}

int cbco_encode_blocked(const cbco_batch *b, const cbco_genome *g, uint32_t L, uint32_t block_reads,
                        uint32_t gen_mode, cbco_buf *out) {
    uint32_t count[CBCG_GEN_MAX], reads[CBCG_GEN_MAX], last = 0, levels = 0;
    if ((gen_mode & CBCG_MODE_GEN_MASK) > 1 || (gen_mode & ~(CBCG_MODE_GEN_MASK | CBCG_MODE_LAYOUT_MASK | CBCG_MODE_REQ_HYBRID))) return -30;
    /* low byte: generations; bit 9: four substreams everywhere; bits 16..23: in that many leading generations; bit 10: the default cut's own choice */
    const uint32_t layout = (gen_mode & CBCG_MODE_SPLIT4) ? 4u : ((gen_mode & CBCG_MODE_REQ_HYBRID) && (gen_mode & CBCG_MODE_GEN_MASK)) ? 0u : 1u;
    uint32_t split_gens = 0;
    if (gen_mode & CBCG_MODE_GEN_MASK) levels = cbcg_gen_schedule(b->n_reads, layout, count, reads, &last, &split_gens);
    if (layout == 0u) gen_mode = (gen_mode & ~CBCG_MODE_REQ_HYBRID) | CBCG_MODE_WITH_SPLIT_GENS(split_gens);
    gen_mode &= ~CBCG_MODE_REQ_HYBRID;
    if (block_reads == 0xffffffffu) block_reads = (gen_mode & CBCG_MODE_GEN_MASK) ? last : 1024u;      /* CBCG_BLOCK_AUTO */
    return encode_cut(b, g, L, block_reads, levels, count, reads, NULL, 0, gen_mode, out);
}

int cbco_decode_blocked(const uint8_t *p, uint64_t len, const cbco_genome *g, cbco_buf *seq_out, uint64_t *n_reads_out) {
    if (len < 40) return -40;
    uint32_t h[10]; memcpy(h, p, 40);
    if (h[0] != CBCG_MAGIC || h[1] != CBCG_VERSION) return -41;
    uint32_t L = h[3]; uint64_t n_reads; memcpy(&n_reads, p + 16, 8);
    uint32_t nb = h[6], n_chr = h[7], gen_mode = h[9] & CBCG_MODE_GEN_MASK;
    const uint32_t fixed_len = (h[9] & CBCG_MODE_FIXED_LEN) ? L : 0;
    if (gen_mode > 1 || (h[9] & ~(CBCG_MODE_GEN_MASK | CBCG_MODE_FIXED_LEN | CBCG_MODE_LAYOUT_MASK)) || n_chr > g->n_chr) return -42;
    if (fixed_len && h[2] != L) return -42;
    uint64_t o = 40;
    /* container chromosome ordinal -> genome ordinal, by name */
    uint32_t *chr_map = (uint32_t *)calloc(n_chr + 1, sizeof(uint32_t));
    for (uint32_t c = 0; c < n_chr; c++) {
        if (o + 4 > len) { free(chr_map); return -43; }
        uint32_t nl; memcpy(&nl, p + o, 4); o += 4;
        if (o + nl > len) { free(chr_map); return -43; }
        uint32_t found = 0xffffffffu;
        for (uint32_t k = 0; k < g->n_chr; k++) if (strlen(g->name[k]) == nl && !memcmp(g->name[k], p + o, nl)) found = k;
        if (found == 0xffffffffu) { free(chr_map); return -44; }
        chr_map[c] = found;
        o += nl + ((4 - (nl & 3)) & 3);
    }
    if (o + 4 > len) { free(chr_map); return -43; }
    uint32_t ix_bytes; memcpy(&ix_bytes, p + o, 4); o += 4;
    if (o + ix_bytes > len || nb > ix_bytes) { free(chr_map); return -43; }
    blk_index *idx = (blk_index *)calloc((size_t)nb + 1, sizeof(blk_index));
    {
        idx_state st = { h[8], 0, 0, 0, 0, 0, { 0, 0, 0, 0 } };
        uint64_t io = o;
        for (uint32_t k = 0; k < nb; k++) if (index_get(p, o + ix_bytes, &io, &st, &idx[k], h[9])) { free(chr_map); free(idx); return -43; }
    }
    o += ix_bytes;
    int rc = 0; uint64_t n = 0;
    uint16_t e[3 * 256 + 8]; uint8_t line[1025];
    uint32_t last_gen = 0, max_block = 0;
    for (uint32_t k = 0; k < nb; k++) { last_gen = idx[k].gen; if (idx[k].n_reads > max_block) max_block = idx[k].n_reads; }   /* the index codes generations in ascending order */
    const uint32_t flag_target = cbcg_flag_target(max_block);
    models *prev = (models *)malloc(sizeof(models)), *acc = NULL;
    models_init(prev, L);
    uint32_t cur_gen = 0;
    for (uint32_t k = 0; k < nb && !rc; k++) {
        blk_index bi; memcpy(&bi, &idx[k], sizeof bi);
        if (bi.chr >= n_chr || o + bi.payload_bytes > len) { rc = -45; break; }
        if (bi.gen != cur_gen) {
            if (acc) { merge_finish(acc, prev, flag_target); models_free(prev); free(prev); prev = acc; acc = NULL; }
            cur_gen = bi.gen;
        }
        if (!acc && bi.gen != last_gen) { acc = (models *)malloc(sizeof(models)); models_clone(acc, prev); }
        uint32_t chr = chr_map[bi.chr];
        rstate s; rstate_init_from(&s, prev, 2);
        s.lean = 1; s.fixed_len = fixed_len;
        const uint32_t n_sub = CBCG_BLOCK_NSUB(h[9], bi.gen);
        s.c.split = n_sub > 1u;
        { uint64_t so = o; for (uint32_t q = 0; q < n_sub; q++) { ac_init_dec(&s.c.ac[q], p + so, bi.sub_bytes[q]); so += bi.sub_bytes[q]; } }
        s.prev_pos = bi.base_pos;
        snp_reset(&s.snp, g->len[chr] + 2048);
        for (uint32_t r = 0; r < bi.n_reads && !rc; r++) {
            cbcg_read_rec rec; uint32_t ne = 0;
            get_read(&s, &rec, e, &ne, g->bases[chr], g->len[chr]);
            if (s.c.err) { rc = s.c.err; break; }
            if (rec.len > 1024 || rebuild_read(&rec, e, g->bases[chr], g->len[chr], line)) { rc = -47; break; }
            line[rec.len] = '\n';
            buf_put(seq_out, line, rec.len + 1u);
            n++;
        }
        if (acc && !rc) merge_block(acc, &s.c.M, prev);
        rstate_free(&s);
        o += bi.payload_bytes;
    }
    if (acc) { models_free(acc); free(acc); }
    models_free(prev); free(prev);
    free(idx);
    free(chr_map);
    if (n_reads_out) *n_reads_out = n;
    return rc;
}
