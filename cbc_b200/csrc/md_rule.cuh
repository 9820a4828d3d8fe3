/* md_rule.cuh -- the one MD rule on the device, shared by K6 (k6_sam.cu: MD of a SAM line's verbatim CIGAR) and K7
 * (k7_md.cu: MD of a read that carries none).
 *
 * The MD of an aligned read is computed from its CIGAR, its SEQ and the reference as uploaded (upper-cased): M, = and X
 * consume read and reference, I and S the read, D the reference, H and P neither. An aligned base is a mismatch when the
 * read base differs from the reference base, so N against N is NOT a mismatch. The spelling is canonical,
 * [0-9]+(([A-Z]|\^[A-Z]+)[0-9]+)*: a number before every event and at the end, 0 included; the letters are reference bases. */
#pragma once
#include <stdint.h>

/* Output cursor: counts only (W false) or counts and writes. */
template <bool W> struct K6Out {
    uint8_t *p; uint32_t n;
    __device__ __forceinline__ void put(uint32_t c) { if (W) p[n] = (uint8_t)c; n++; }
    __device__ __forceinline__ void num(uint32_t v) {
        const uint32_t d = v >= 1000000000u ? 10u : v >= 100000000u ? 9u : v >= 10000000u ? 8u : v >= 1000000u ? 7u : v >= 100000u ? 6u
                         : v >= 10000u ? 5u : v >= 1000u ? 4u : v >= 100u ? 3u : v >= 10u ? 2u : 1u;
        if (W) for (uint32_t j = d; j-- > 0u;) { p[n + j] = (uint8_t)('0' + v % 10u); v /= 10u; }
        n += d;
    }
    __device__ __forceinline__ void str(const char *s) { for (; *s; s++) put((uint8_t)*s); }
    __device__ __forceinline__ void cig(uint32_t cnt, uint32_t op) { num(cnt); put(op); }   /* one CIGAR operation as text */
};

/* Verbatim CIGAR: true when its read length is len, it deletes at most K6_MAX_DEL bases (what the host's size bound and the
   reference's pad allow for) and its operations are M I D S H P = X only. */
#define K6_MAX_DEL 255u
__device__ static bool k6_cigar_ok(const uint8_t *t, uint32_t tl, uint32_t len) {
    uint32_t i = 0, q = 0, d = 0;
    while (i < tl) {
        uint32_t num = 0, digits = 0;
        while (i < tl && t[i] >= '0' && t[i] <= '9' && digits < 10u) { num = num * 10u + (uint32_t)(t[i] - '0'); i++; digits++; }
        if (!digits || digits > 9u || i >= tl) return false;
        const uint32_t op = t[i++];
        if (op == 'M' || op == '=' || op == 'X' || op == 'I' || op == 'S') { q += num; if (q > len) return false; }
        else if (op == 'D') { d += num; if (d > K6_MAX_DEL) return false; }
        else if (op != 'H' && op != 'P') return false;
    }
    return q == len;
}

/* MD of the general path: the CIGAR text walked against SEQ and the reference; *nm receives NM. The CIGAR must have passed
   k6_cigar_ok: the walk reads seq[0, len) and ref[0, M + = + X + D) and nothing else. */
template <bool W> __device__ static void k6_md_walk(K6Out<W> &o, const uint8_t *t, uint32_t tl, const uint8_t *seq, const uint8_t *ref,
                                                    uint32_t *nm) {
    uint32_t i = 0, ri = 0, rp = 0, run = 0, n = 0;
    while (i < tl) {
        uint32_t num = 0;
        while (t[i] >= '0' && t[i] <= '9') num = num * 10u + (uint32_t)(t[i++] - '0');
        const uint32_t op = t[i++];
        if (op == 'M' || op == '=' || op == 'X') {
            for (uint32_t j = 0; j < num; j++, ri++, rp++) {
                const uint32_t rb = ref[rp];
                if (seq[ri] != rb) { o.num(run); o.put(rb); run = 0; n++; } else run++;
            }
        } else if (op == 'I') { ri += num; n += num; }
        else if (op == 'S') ri += num;
        else if (op == 'D') {
            o.num(run); o.put('^');
            for (uint32_t j = 0; j < num; j++) o.put(ref[rp++]);
            run = 0; n += num;
        }
    }
    o.num(run);
    *nm = n;
}
