/* sam_fields.cuh -- the fields of an alignment record that the device derives from a decoded record, shared by K6
 * (k6_sam.cu: SAM text) and K9 (k9_bam.cu: BAM records), so that both formats carry one CIGAR, MD and NM. The MD rule and
 * the verbatim CIGAR's checks and walk are md_rule.cuh's (shared with K7). */
#pragma once
#include "common.cuh"
#include "md_rule.cuh"

/* The implied CIGAR (k4_cigar.cu, cig_implied) streamed op by op, one op late so that the last one is known; the first
   and last I become S per the class. Each op goes to o.cig(count, op letter): SAM text for K6, a BAM u32 for K9. Returns
   the bases of I operations that stay I (for NM). */
template <class Out> __device__ static uint32_t k6_cigar_implied(Out &o, uint32_t len, uint32_t nd, uint32_t ni, const uint16_t *dels,
                                                              const uint16_t *ins, uint32_t cls) {
    const uint32_t total_m = len - ni;
    uint32_t cur = 0, kd = 0, ki = 0, dc = 0, ic = 0, k = 0, ins_bases = 0;
    uint32_t pend = 0;                                   /* (count << 8 | op) not yet written; 0: none */
    auto emit = [&](uint32_t op, bool last) {
        uint32_t c = op & 0xffu;
        const uint32_t cnt = op >> 8;
        if (c == 'I' && ((k == 0u && (cls & 1u)) || (last && k != 0u && (cls & 2u)))) c = 'S';
        if (c == 'I') ins_bases += cnt;
        o.cig(cnt, c); k++;
    };
    auto push = [&](uint32_t op) { if (pend) emit(pend, false); pend = op; };
    while (kd < nd || ki < ni) {
        const uint32_t dn = kd < nd ? dc + CBCG_EDIT_DELTA(dels[kd]) : 0xffffffffu;
        const uint32_t in = ki < ni ? ic + CBCG_EDIT_DELTA(ins[ki]) : 0xffffffffu;
        const uint32_t at = min(dn, in);
        if (at > cur) { push(((at - cur) << 8) | 'M'); cur = at; }
        if (in == at) {
            uint32_t q = 0;
            while (ki < ni && ic + CBCG_EDIT_DELTA(ins[ki]) == at) { ic = at; ki++; q++; }
            push((q << 8) | 'I');
        }
        if (dn == at) {
            uint32_t q = 0;
            while (kd < nd && dc + CBCG_EDIT_DELTA(dels[kd]) == at) { dc = at; kd++; q++; }
            push((q << 8) | 'D');
        }
    }
    if (total_m > cur) push(((total_m - cur) << 8) | 'M');
    if (pend) emit(pend, true);
    return ins_bases;
}

/* MD of the fast path from the SNP and deletion lists; returns the mismatches. ref: the read's reference, from its POS.
   An event beyond the read (a record K1 does not write; K3 reports it) ends the walk: *bad is set. */
template <bool W> __device__ static uint32_t k6_md_edits(K6Out<W> &o, uint32_t total_m, uint32_t nd, uint32_t ns, const uint16_t *dels,
                                                         const uint16_t *snps, const uint8_t *ref, bool *bad) {
    uint32_t last = 0, kd = 0, ks = 0, dc = 0, s_next = 0, dels_before = 0, mis = 0;
    while (kd < nd || ks < ns) {
        const uint32_t d_at = kd < nd ? dc + CBCG_EDIT_DELTA(dels[kd]) : 0xffffffffu;
        const uint32_t s_at = ks < ns ? s_next + CBCG_EDIT_DELTA(snps[ks]) : 0xffffffffu;   /* SNP k sits at sum_{i<k}(p_i + 1) + p_k */
        if (d_at <= s_at ? d_at > total_m : s_at >= total_m) { *bad = true; break; }
        if (d_at <= s_at) {                               /* a deletion at coordinate a comes before aligned base a */
            o.num(d_at - last); o.put('^');
            while (kd < nd && dc + CBCG_EDIT_DELTA(dels[kd]) == d_at) { dc = d_at; kd++; o.put(ref[d_at + dels_before]); dels_before++; }
            last = d_at;
        } else {
            const uint32_t rb = ref[s_at + dels_before], qb = base_char(CBCG_EDIT_TARGET(snps[ks]));
            if (qb != rb) { o.num(s_at - last); o.put(rb); last = s_at + 1u; mis++; }
            s_next = s_at + 1u; ks++;
        }
    }
    o.num(total_m > last ? total_m - last : 0u);
    return mis;
}
