/*
 * k8_pileup.cu -- K8: per-position base, deletion and insertion counts over regions (cbcg_pileup).
 *
 * Runs on the reads the region decode kept (K5: records, chromosome ordinals, container ordinals) and, only when the
 * CIGAR side section lists class-4 reads, on K3's text (SEQ + '\n' per read). Every read is aligned by the CIGAR its SAM
 * line carries (k6_sam.cu): the implied CIGAR for classes 0..3, the section's verbatim text for class 4.
 *
 *   accumulators: one slot per reference position of the merged request intervals (api.cu: sorted by (chromosome,
 *     start), overlapping and adjacent ones merged, clipped to the record's length), plus one slot after each interval
 *     that takes the -1 of a run ending at the interval's last position. Eight u32 columns of n_pad slots each (n_pad a
 *     multiple of K8_SCAN_TILE, zeroed by the host): cov_diff, del_diff, then the SNP-base counts A C G T N, then INS.
 *   scatter: one thread per read, tiles of K8_TILE from an atomic ticket. A read with FLAG & flag_exclude is skipped.
 *     fast path (classes 0..3): the deletion and insertion lists give the aligned runs (cig_implied's walk, I before D at
 *     one coordinate); a run clipped to an interval adds +1 / -1 to cov_diff, a deletion run the same to del_diff; a SNP
 *     adds one to its target base's count (its coordinate is the format's sum_{i<k}(p_i + 1) + p_k, shifted by the
 *     deletions at or before it, as in k6_md_edits); an insertion run whose coordinate has aligned bases on both sides
 *     adds one to INS at the last reference position before it. No base of the read is read: every aligned base that is
 *     not a SNP is the reference base.
 *     general path (class 4): the verbatim CIGAR walked against SEQ; an aligned base whose code differs from the
 *     reference base's counts like a SNP. An I operation with an M / = / X before and after it counts once per reference
 *     position.
 *   scan: an in-place inclusive scan of cov_diff and del_diff (a CTA scan and a decoupled look-back per column). Each
 *     interval's slots, its extra slot included, sum to zero, so one scan over all intervals needs no reset. A tile's
 *     total can be negative: the look-back carries it biased by K8_BIAS (|total| <= reads, < 2^32).
 *   gather: one thread per output row (binary search over the regions' row offsets): A C G T N DEL INS REF, where the
 *     reference base's column is depth - sum(SNP counts) + its own SNP count.
 *
 * Every index into the accumulators and the genome is checked on the device; a record that fails a check sets the
 * error word and writes nothing.
 */
#include "common.cuh"
#include "internal.h"
#include "md_rule.cuh"

#define K8_TILE 128u
#define K8_SCAN_THREADS 256u
#define K8_SCAN_PER 4u
#define K8_GATHER 256u
#define K8_BIAS (1ull << 33)

uint64_t pileup_num_tiles(uint64_t n_reads) { return (n_reads + K8_TILE - 1u) / K8_TILE; }


struct K8Acc {
    uint32_t *a; uint64_t n_pad;
    __device__ __forceinline__ void add(uint32_t col, uint64_t slot, uint32_t v) const { atomicAdd(a + col * n_pad + slot, v); }
};

/* One interval's view of a read: slots of reference positions [s, e] start at slot0; slot0 + (e - s) + 1 is the extra slot. */
struct K8Iv {
    uint64_t s, e, slot0;
    __device__ __forceinline__ void run(const K8Acc &A, uint32_t col, uint64_t x, uint64_t y) const {   /* [x, y], 1-based */
        const uint64_t lo = max(x, s), hi = min(y, e);
        if (x > y || lo > hi) return;
        A.add(col, slot0 + (lo - s), 1u);
        A.add(col, slot0 + (hi - s) + 1u, 0xffffffffu);
    }
    __device__ __forceinline__ void one(const K8Acc &A, uint32_t col, uint64_t p) const {
        if (p >= s && p <= e) A.add(col, slot0 + (p - s), 1u);
    }
};

/* Fast path. Returns false when an edit lies beyond the read (nothing is written then: the checks come first). */
__device__ static bool k8_edits_ok(uint32_t aligned, uint32_t nd, uint32_t ns, uint32_t ni, const uint16_t *e) {
    uint32_t c = 0;
    for (uint32_t k = 0; k < nd; k++) c += CBCG_EDIT_DELTA(e[k]);
    if (nd && c > aligned) return false;
    c = 0;
    for (uint32_t k = 0; k < ns; k++) { c += CBCG_EDIT_DELTA(e[nd + k]) + (k ? 1u : 0u); if (c >= aligned) return false; }
    c = 0;
    for (uint32_t k = 0; k < ni; k++) c += CBCG_EDIT_DELTA(e[nd + ns + k]);
    return !(ni && c > aligned);
}

__device__ static void k8_fast(const K8Acc &A, const K8Iv &V, uint64_t pos, uint32_t aligned, uint32_t nd, uint32_t ns, uint32_t ni,
                               const uint16_t *dels, const uint16_t *snps, const uint16_t *ins) {
    /* aligned runs, deletion runs and interior insertions */
    uint64_t rp = pos;                                   /* next reference position */
    uint32_t cur = 0, kd = 0, ki = 0, dc = 0, ic = 0;
    while (kd < nd || ki < ni) {
        const uint32_t dn = kd < nd ? dc + CBCG_EDIT_DELTA(dels[kd]) : 0xffffffffu;
        const uint32_t in = ki < ni ? ic + CBCG_EDIT_DELTA(ins[ki]) : 0xffffffffu;
        const uint32_t at = min(dn, in);
        if (at > cur) { V.run(A, 0, rp, rp + (at - cur) - 1u); rp += at - cur; cur = at; }
        if (in == at) {
            while (ki < ni && ic + CBCG_EDIT_DELTA(ins[ki]) == at) { ic = at; ki++; }
            if (at > 0u && at < aligned) V.one(A, 7, rp - 1u);
        }
        if (dn == at) {
            uint32_t q = 0;
            while (kd < nd && dc + CBCG_EDIT_DELTA(dels[kd]) == at) { dc = at; kd++; q++; }
            V.run(A, 1, rp, rp + q - 1u); rp += q;
        }
    }
    if (aligned > cur) V.run(A, 0, rp, rp + (aligned - cur) - 1u);
    /* SNPs: aligned coordinate plus the deletions at or before it */
    uint32_t kd2 = 0, dc2 = 0, s_next = 0;
    for (uint32_t k = 0; k < ns; k++) {
        const uint32_t s_at = s_next + CBCG_EDIT_DELTA(snps[k]);
        while (kd2 < nd && dc2 + CBCG_EDIT_DELTA(dels[kd2]) <= s_at) { dc2 += CBCG_EDIT_DELTA(dels[kd2]); kd2++; }
        const uint32_t t = CBCG_EDIT_TARGET(snps[k]);
        V.one(A, 2u + min(t, 4u), pos + s_at + kd2);
        s_next = s_at + 1u;
    }
}

/* General path over a CIGAR that passed k6_cigar_ok (so seq[0, len) and ref[0, M + = + X + D) are the only bytes read). */
__device__ static void k8_general(const K8Acc &A, const K8Iv &V, uint64_t pos, const uint8_t *t, uint32_t tl, const uint8_t *seq,
                                  const uint8_t *ref) {
    /* the end of the last aligned operation (of at least one base): an I after it has no aligned base after it */
    uint32_t last_m = 0;
    for (uint32_t i = 0; i < tl;) {
        uint32_t num = 0;
        while (t[i] >= '0' && t[i] <= '9') num = num * 10u + (uint32_t)(t[i++] - '0');
        const uint32_t op = t[i++];
        if ((op == 'M' || op == '=' || op == 'X') && num) last_m = i;
    }
    uint64_t rp = pos, last_ins = 0;
    uint32_t ri = 0;
    bool seen_m = false;
    for (uint32_t i = 0; i < tl;) {
        uint32_t num = 0;
        while (t[i] >= '0' && t[i] <= '9') num = num * 10u + (uint32_t)(t[i++] - '0');
        const uint32_t op = t[i++];
        if (op == 'M' || op == '=' || op == 'X') {
            V.run(A, 0, rp, rp + num - 1u);
            const uint64_t lo = max(rp, V.s), hi = min(rp + num - 1u, V.e);
            for (uint64_t p = lo; num && p <= hi; p++) {
                const uint32_t qb = base_code(seq[ri + (uint32_t)(p - rp)]);
                if (qb != base_code(ref[p - pos])) A.add(2u + qb, V.slot0 + (p - V.s), 1u);
            }
            ri += num; rp += num; seen_m |= num != 0u;
        } else if (op == 'I') {
            if (seen_m && i < last_m && num && rp - 1u != last_ins) { V.one(A, 7, rp - 1u); last_ins = rp - 1u; }
            ri += num;
        } else if (op == 'S') ri += num;
        else if (op == 'D') { V.run(A, 1, rp, rp + num - 1u); rp += num; }
    }
}

__global__ void __launch_bounds__(K8_TILE)
k8_scatter_kernel(uint64_t n_reads, const cbcg_read_rec *__restrict__ recs, const uint32_t *__restrict__ chr_of,
                  const uint16_t *__restrict__ edits, DevGenome g, const RegionIv *__restrict__ iv, const uint64_t *__restrict__ iv_slot,
                  uint32_t n_iv, uint32_t flag_exclude, const uint64_t *__restrict__ ids, const uint8_t *__restrict__ cls,
                  const uint64_t *__restrict__ exc_read, const uint64_t *__restrict__ exc_off, const uint8_t *__restrict__ exc_text,
                  uint64_t n_exc, const uint8_t *__restrict__ seq_text, uint32_t max_len, uint32_t fixed_len, uint64_t *desc_seq,
                  uint32_t *acc, uint64_t n_pad, uint64_t n_slots, uint32_t *ticket, uint64_t *n_counted, unsigned long long *err) {
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp[K8_TILE / 32u];
    __shared__ uint64_t s_seq_base;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t r0 = (uint64_t)tile * K8_TILE, r = r0 + tid;
    const uint32_t nr = (uint32_t)min((uint64_t)K8_TILE, n_reads - r0);

    cbcg_read_rec rec;
    uint32_t chr = 0, seq_bytes = 0;
    bool live = false, bad = true;
    const uint8_t *verb = nullptr; uint32_t verb_len = 0;
    if (tid < nr) {
        *reinterpret_cast<uint4 *>(&rec) = reinterpret_cast<const uint4 *>(recs)[r];
        chr = chr_of[r];
        const uint32_t len = rec.len, pos = rec.pos;
        const bool bad_len = len == 0u || len > max_len || (fixed_len && len != fixed_len);
        bad = bad_len || pos == 0u || chr >= g.n_chr || (uint64_t)(pos - 1u) > g.chr_len[chr] || (!rec.match && rec.n_ins > len);
        seq_bytes = bad_len ? 1u : len + 1u;
        if (bad) dev_set_error(err, CBCG_ERR_CORRUPT, r);
        else if (!(rec.flag & flag_exclude)) {
            live = true;
            if (cls) {
                const uint64_t ord = ids ? ids[r] : r;
                if (cls[ord] >= 4u) {                       /* verbatim: its entry by binary search over the listed reads */
                    uint64_t lo = 0, hi = n_exc;
                    while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (exc_read[mid] < ord) lo = mid + 1; else hi = mid; }
                    if (lo < n_exc && exc_read[lo] == ord && seq_text &&
                        k6_cigar_ok(exc_text + exc_off[lo], (uint32_t)(exc_off[lo + 1] - exc_off[lo]), len)) {
                        verb = exc_text + exc_off[lo]; verb_len = (uint32_t)(exc_off[lo + 1] - exc_off[lo]);
                    } else { dev_set_error(err, CBCG_ERR_FORMAT, r); live = false; }
                }
            }
        }
    }
    const uint32_t n_live = __syncthreads_count(live);
    if (tid == 0 && n_live) atomicAdd(reinterpret_cast<unsigned long long *>(n_counted), (unsigned long long)n_live);

    /* the read's SEQ in K3's text: only the general path reads it */
    uint64_t seq_at = 0;
    if (seq_text) {
        const uint32_t incl = warp_incl_scan(seq_bytes);
        if (lane == 31u) s_warp[warp] = incl;
        __syncthreads();
        uint32_t warp_base = 0, total = 0;
#pragma unroll
        for (uint32_t k = 0; k < K8_TILE / 32u; k++) { const uint32_t t = s_warp[k]; if (k < warp) warp_base += t; total += t; }
        if (fixed_len) { if (tid == 0) s_seq_base = r0 * (uint64_t)(fixed_len + 1u); }
        else if (warp == 0) { const uint64_t b = lookback_exclusive(desc_seq, tile, total, err); if (lane == 0) s_seq_base = b; }
        __syncthreads();
        seq_at = s_seq_base + warp_base + incl - seq_bytes;
    }
    if (!live) return;

    const uint32_t len = rec.len;
    const uint64_t pos = rec.pos;
    const uint32_t nd = rec.match ? 0u : rec.n_dels, ns = rec.match ? 0u : rec.n_snps, ni = rec.match ? 0u : rec.n_ins;
    const uint32_t aligned = len - ni;
    const uint16_t *e = edits + rec.edit_off;
    uint64_t last;                                       /* the read's last reference position, for the interval search */
    if (verb) {
        uint32_t span = 0;
        for (uint32_t i = 0; i < verb_len;) {
            uint32_t num = 0;
            while (verb[i] >= '0' && verb[i] <= '9') num = num * 10u + (uint32_t)(verb[i++] - '0');
            const uint32_t op = verb[i++];
            if (op == 'M' || op == '=' || op == 'X' || op == 'D') span += num;
        }
        last = pos + (span ? span : 1u) - 1u;
    } else {
        if (!k8_edits_ok(aligned, nd, ns, ni, e)) { dev_set_error(err, CBCG_ERR_CORRUPT, r); return; }
        last = pos + (aligned + nd ? aligned + nd : 1u) - 1u;
    }
    const K8Acc A{ acc, n_pad };
    const uint8_t *ref = g.bases + g.chr_off[chr] + (pos - 1u);
    /* the first interval of this chromosome that ends at or after pos, then every one that starts by the read's end */
    uint32_t lo = 0, hi = n_iv;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const RegionIv v = iv[mid];
        if (v.chr < chr || (v.chr == chr && v.end < pos)) lo = mid + 1u; else hi = mid;
    }
    for (uint32_t j = lo; j < n_iv && iv[j].chr == chr && iv[j].start <= last; j++) {
        const K8Iv V{ iv[j].start, iv[j].end, iv_slot[j] };
        if (V.e < V.s || V.slot0 + (V.e - V.s) + 1u >= n_slots || V.e > g.chr_len[chr]) { dev_set_error(err, CBCG_ERR_INTERNAL, r); return; }
        if (verb) k8_general(A, V, pos, verb, verb_len, seq_text + seq_at, ref);
        else k8_fast(A, V, pos, aligned, nd, ns, ni, e, e + nd, e + nd + ns);
    }
}

__global__ void __launch_bounds__(K8_SCAN_THREADS)
k8_scan_kernel(uint32_t *acc, uint64_t n_pad, uint64_t *desc, uint32_t *ticket, unsigned long long *err) {
    __shared__ uint32_t s_tile;
    __shared__ int32_t s_warp[2][K8_SCAN_THREADS / 32u];
    __shared__ int64_t s_base[2];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t n_tiles = n_pad / K8_SCAN_TILE;
    const uint64_t at = (uint64_t)tile * K8_SCAN_TILE + (uint64_t)tid * K8_SCAN_PER;
    int4 v[2];
    int32_t mine[2], incl[2];
#pragma unroll
    for (uint32_t c = 0; c < 2u; c++) {
        v[c] = *reinterpret_cast<const int4 *>(acc + c * n_pad + at);
        v[c].y += v[c].x; v[c].z += v[c].y; v[c].w += v[c].z;
        mine[c] = v[c].w;
        /* warp inclusive scan of signed values (two's complement: the unsigned scan gives the same bits) */
        incl[c] = (int32_t)warp_incl_scan((uint32_t)mine[c]);
        if (lane == 31u) s_warp[c][warp] = incl[c];
    }
    __syncthreads();
    int64_t wbase[2] = { 0, 0 }, total[2] = { 0, 0 };
#pragma unroll
    for (uint32_t c = 0; c < 2u; c++)
#pragma unroll
        for (uint32_t k = 0; k < K8_SCAN_THREADS / 32u; k++) { const int64_t t = s_warp[c][k]; if (k < warp) wbase[c] += t; total[c] += t; }
    if (warp < 2u) {                                     /* warp 0: cov_diff, warp 1: del_diff */
        const int64_t mine_total = warp ? total[1] : total[0];
        const uint64_t b = lookback_exclusive(desc + warp * n_tiles, tile, (uint64_t)(mine_total + (int64_t)K8_BIAS), err);
        if (lane == 0) s_base[warp] = (int64_t)(b - (uint64_t)tile * K8_BIAS);
    }
    __syncthreads();
#pragma unroll
    for (uint32_t c = 0; c < 2u; c++) {
        const int64_t base = s_base[c] + wbase[c] + incl[c] - mine[c];
        int4 o;
        o.x = (int32_t)(base + v[c].x); o.y = (int32_t)(base + v[c].y); o.z = (int32_t)(base + v[c].z); o.w = (int32_t)(base + v[c].w);
        if (base + min(min(v[c].x, v[c].y), min(v[c].z, v[c].w)) < 0) dev_set_error(err, CBCG_ERR_INTERNAL, at);
        *reinterpret_cast<int4 *>(acc + c * n_pad + at) = o;
    }
}

/* rows: n_rows x 8 u32. reg: per region, { first row, chromosome, first position, first slot } (n_reg of them, ascending
   first row). */
__global__ void __launch_bounds__(K8_GATHER)
k8_gather_kernel(uint64_t n_rows, const PileupReg *__restrict__ reg, uint32_t n_reg, const uint32_t *__restrict__ acc, uint64_t n_pad,
                 uint64_t n_slots, DevGenome g, uint32_t *__restrict__ rows, unsigned long long *err) {
    const uint64_t t = (uint64_t)blockIdx.x * K8_GATHER + threadIdx.x;
    if (t >= n_rows) return;
    uint32_t lo = 0, hi = n_reg;                         /* the last region whose first row is at or below t */
    while (hi - lo > 1u) { const uint32_t mid = (lo + hi) >> 1; if (reg[mid].row0 <= t) lo = mid; else hi = mid; }
    const PileupReg R = reg[lo];
    const uint64_t k = t - R.row0, p = R.start + k, slot = R.slot0 + k;
    if (R.row0 > t || slot >= n_slots || R.chr >= g.n_chr || p == 0u || p > g.chr_len[R.chr]) { dev_set_error(err, CBCG_ERR_INTERNAL, t); return; }
    const int32_t depth = (int32_t)acc[slot], del = (int32_t)acc[n_pad + slot];
    uint32_t s[5], sum = 0;
#pragma unroll
    for (uint32_t b = 0; b < 5u; b++) { s[b] = acc[(2u + b) * n_pad + slot]; sum += s[b]; }
    const uint32_t refb = g.bases[g.chr_off[R.chr] + (p - 1u)];
    if (depth < 0 || del < 0 || (uint32_t)depth < sum) { dev_set_error(err, CBCG_ERR_INTERNAL, t); return; }
    s[base_code(refb)] += (uint32_t)depth - sum;
    uint4 *o = reinterpret_cast<uint4 *>(rows + t * CBCG_PU_COLS);
    o[0] = make_uint4(s[0], s[1], s[2], s[3]);
    o[1] = make_uint4(s[4], (uint32_t)del, acc[7u * n_pad + slot], refb);
}

int launch_pileup(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const uint16_t *edits, const DevGenome &g,
                  const RegionIv *iv, const uint64_t *iv_slot, uint32_t n_iv, uint32_t flag_exclude, const uint64_t *ids, const uint8_t *cls,
                  const uint64_t *exc_read, const uint64_t *exc_off, const uint8_t *exc_text, uint64_t n_exc, const uint8_t *seq_text,
                  uint32_t max_len, uint32_t fixed_len, uint32_t *acc, uint64_t n_pad, uint64_t n_slots, const PileupReg *reg, uint32_t n_reg,
                  uint32_t *rows, uint64_t n_rows, uint64_t *tile_desc, uint32_t *ticket, uint64_t *n_counted, unsigned long long *err,
                  cudaStream_t st) {
    if (n_pad % K8_SCAN_TILE || n_slots > n_pad) return -1;
    if (cudaMemsetAsync(n_counted, 0, sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (n_reads) {
        const uint64_t tiles = pileup_num_tiles(n_reads);
        if (cudaMemsetAsync(tile_desc, 0, tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
        if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
        k8_scatter_kernel<<<(unsigned)tiles, K8_TILE, 0, st>>>(n_reads, recs, chr, edits, g, iv, iv_slot, n_iv, flag_exclude, ids, cls,
                                                               exc_read, exc_off, exc_text, n_exc, seq_text, max_len, fixed_len, tile_desc,
                                                               acc, n_pad, n_slots, ticket, n_counted, err);
        if (cudaGetLastError() != cudaSuccess) return -1;
    }
    if (n_pad) {
        const uint64_t tiles = n_pad / K8_SCAN_TILE;
        if (cudaMemsetAsync(tile_desc, 0, 2u * tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
        if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
        k8_scan_kernel<<<(unsigned)tiles, K8_SCAN_THREADS, 0, st>>>(acc, n_pad, tile_desc, ticket, err);
        if (cudaGetLastError() != cudaSuccess) return -1;
    }
    if (n_rows) {
        k8_gather_kernel<<<(unsigned)((n_rows + K8_GATHER - 1u) / K8_GATHER), K8_GATHER, 0, st>>>(n_rows, reg, n_reg, acc, n_pad, n_slots, g,
                                                                                                  rows, err);
        if (cudaGetLastError() != cudaSuccess) return -1;
    }
    return 0;
}
