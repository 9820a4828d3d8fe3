/*
 * k6_sam.cu -- K6: SAM alignment records (cbcg_decode_sam).
 *
 * Runs after K3, over K3's text (SEQ + '\n' per read) and the records the block decoder wrote (or K5 kept). One line
 * per read, in the order of the records:
 *
 *   *  FLAG  RNAME  POS  255  CIGAR  *  0  0  SEQ  *  NM:i:<n>  MD:Z:<md>
 *
 * QNAME, MAPQ, the mate fields and QUAL are not stored by the format: they carry the SAM spec's "unavailable" values.
 *
 *   CIGAR: class 0..3 (no side section: every read is class 0) -- the CIGAR the deletions and insertions imply, merged
 *     as in k4_cigar.cu's cig_implied, with the first / the last end operation turned from I into S per the class;
 *     class 4 -- the side section's verbatim text.
 *   MD and NM are recomputed from the line's own CIGAR, its SEQ and the reference as uploaded (upper-cased; the rule is
 *     md_rule.cuh's, which K7 shares):
 *     M, = and X consume read and reference, I and S the read, D the reference, H and P neither. An aligned base is a
 *     mismatch when the read base differs from the reference base, so N against N is NOT a mismatch (samtools calmd
 *     counts it as one; here a base that equals the reference is a match whatever it is). MD is spelled canonically,
 *     [0-9]+(([A-Z]|\^[A-Z]+)[0-9]+)*: a number before every event and at the end, 0 included; the letters are reference
 *     bases. NM = mismatches + I bases + D bases (clipped bases do not count).
 *   fast path (class 0..3): every aligned base that is not a SNP equals the reference by construction (K3 copied it from
 *     there), so MD and NM follow from the edit list alone, with reference look-ups at the SNP and deletion sites only.
 *     A SNP whose base equals the reference base (N over N) is a match.
 *   general path (class 4: =, X, H, P, or a match record whose input CIGAR was not <len>M, such as a trailing clip over
 *     bases that equal the reference): the CIGAR text is walked against SEQ and the reference. Its deletions need not be
 *     the record's (a read whose bases also equal the reference read straight on, such as 97M2D3M over a repeat, is coded as a perfect match). A text whose read
 *     length is not the record's, that deletes more than 255 bases or that holds another operation is CBCG_ERR_FORMAT
 *     (the line then takes the implied CIGAR, so that its size stays bounded).
 *
 * B200 design. One CTA per tile of K6_TILE consecutive reads, a thread per read. The tile's SEQ is one contiguous range
 * of K3's text (closed-form offset r (L + 1) for CBCG_MODE_FIXED_LEN, otherwise a CTA scan of len + 1 and a decoupled
 * look-back), staged into shared memory by one TMA bulk copy. Each thread sizes its line exactly (a counting pass of
 * the same formatter that writes it), a CTA scan and a second decoupled look-back over line sizes give the output
 * offsets (tile order from an atomic ticket, as K1 / K3 / K4 / K5), the threads write their lines into a shared-memory
 * image, the warps copy the SEQ fields into it, and the image leaves with one TMA bulk store (16-byte aligned middle)
 * plus byte stores for the ragged ends, as K3's does. A tile whose lines do not fit the image (long names, very long
 * CIGAR texts) is written straight to HBM by its threads.
 */
#include "common.cuh"
#include "internal.h"
#include "sam_fields.cuh"

#define K6_TILE 128u

uint64_t sam_num_tiles(uint64_t n_reads) { return (n_reads + K6_TILE - 1u) / K6_TILE; }

/* image bytes per read of the tile: SEQ + '\n' and room for the other fields of an ordinary read */
#define K6_IMG_EXTRA 128u
static inline CBCG_HD uint32_t k6_img_cap(uint32_t max_len) { return K6_TILE * (max_len + 1u + K6_IMG_EXTRA); }
static inline CBCG_HD uint32_t k6_stage_cap(uint32_t max_len) { return ((K6_TILE * (max_len + 1u) + 32u + 15u) & ~15u); }

struct K6Smem {
    uint64_t bar;
    uint64_t seq_base, out_base;
    uint32_t tile;
    uint32_t warp_tot[K6_TILE / 32u], warp_tot2[K6_TILE / 32u];
    uint32_t line_off[K6_TILE];       /* byte offset of each line in the tile */
    uint32_t seq_at[K6_TILE];         /* offset of each read's SEQ field in its line */
    uint32_t seq_src[K6_TILE];        /* offset of each read's SEQ in the stage */
    uint16_t len[K6_TILE];
    __align__(16) uint8_t dyn[16];    /* stage (k6_stage_cap), then the image (k6_img_cap + 32): dynamic */
};

struct K6Read {
    cbcg_read_rec rec;
    uint32_t chr, cls, bad;
    const uint8_t *verb; uint32_t verb_len;            /* class 4 with a valid text */
};

/* One line. Counting pass (W false): returns its size, NM in *nm and whether the edit list runs past the read in *bad.
   Writing pass: nm is given, SEQ is copied from seq when copy_seq (else left for the warps), *seq_at receives the SEQ
   field's offset. */
template <bool W> __device__ static uint32_t k6_line(uint8_t *dst, const K6Read &R, const uint16_t *edits, const DevGenome &g,
                                                     const uint8_t *names, const uint32_t *name_len, const uint8_t *seq, bool copy_seq,
                                                     uint32_t *nm, uint32_t *seq_at, bool *bad) {
    K6Out<W> o{ dst, 0u };
    const cbcg_read_rec &r = R.rec;
    const uint32_t len = r.len;
    o.put('*'); o.put('\t'); o.num(r.flag); o.put('\t');
    if (!R.bad) {
        const uint8_t *nmp = names + (uint64_t)R.chr * MAX_NAME;
        const uint32_t nl = name_len[R.chr];
        for (uint32_t j = 0; j < nl; j++) o.put(nmp[j]);
    } else o.put('*');
    o.put('\t'); o.num(r.pos); o.str("\t255\t");
    const uint32_t nd = r.match ? 0u : r.n_dels, ns = r.match ? 0u : r.n_snps, ni = r.match ? 0u : r.n_ins;
    const uint16_t *e = edits + r.edit_off;
    const uint8_t *ref = R.bad ? nullptr : g.bases + g.chr_off[R.chr] + (r.pos - 1u);
    uint32_t ins_bases = 0;
    if (R.bad) o.put('*');
    else if (R.verb) for (uint32_t j = 0; j < R.verb_len; j++) o.put(R.verb[j]);
    else ins_bases = k6_cigar_implied(o, len, nd, ni, e, e + nd + ns, R.cls);
    o.str("\t*\t0\t0\t");
    *seq_at = o.n;
    if (W && copy_seq) for (uint32_t j = 0; j < len; j++) o.p[o.n + j] = seq[j];
    o.n += len;
    o.str("\t*\tNM:i:");
    /* MD follows NM in the line but is what NM is computed from: the counting pass walks it into a sink first */
    uint32_t n = 0;
    bool malformed = false;
    if (!W) {
        K6Out<false> sink{ nullptr, 0u };
        if (R.bad) n = 0;
        else if (R.verb) k6_md_walk(sink, R.verb, R.verb_len, seq, ref, &n);
        else n = k6_md_edits(sink, len - ni, nd, ns, e, e + nd, ref, &malformed) + ins_bases + nd;
        *nm = n;
    } else n = *nm;
    o.num(n); o.str("\tMD:Z:");
    if (R.bad) o.put('0');
    else if (R.verb) { uint32_t dummy; k6_md_walk(o, R.verb, R.verb_len, seq, ref, &dummy); }
    else k6_md_edits(o, len - ni, nd, ns, e, e + nd, ref, &malformed);
    *bad = malformed;
    o.put('\n');
    return o.n;
}

__global__ void __launch_bounds__(K6_TILE)
k6_sam_kernel(uint64_t n_reads, const cbcg_read_rec *__restrict__ recs, const uint32_t *__restrict__ chr_of, const uint16_t *__restrict__ edits,
              DevGenome g, const uint8_t *__restrict__ names, const uint32_t *__restrict__ name_len, const uint8_t *__restrict__ seq_text,
              uint32_t max_len, uint32_t fixed_len, const uint64_t *__restrict__ ids, const uint8_t *__restrict__ cls,
              const uint64_t *__restrict__ exc_read, const uint64_t *__restrict__ exc_off, const uint8_t *__restrict__ exc_text, uint64_t n_exc,
              uint8_t *__restrict__ out, uint64_t out_cap, uint64_t *desc_seq, uint64_t *desc_out, uint32_t *ticket, uint64_t *total_bytes,
              unsigned long long *err) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    K6Smem &S = *reinterpret_cast<K6Smem *>(smem_raw);
    uint8_t *const s_seq = S.dyn, *const s_img = S.dyn + k6_stage_cap(max_len);
    const uint32_t img_cap = k6_img_cap(max_len);
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) {
        S.tile = atomicAdd(ticket, 1u);
        mbar_init(&S.bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    const uint32_t tile = S.tile;
    const uint64_t r0 = (uint64_t)tile * K6_TILE, r = r0 + tid;
    const uint32_t nr = (uint32_t)min((uint64_t)K6_TILE, n_reads - r0);

    K6Read R;
    R.verb = nullptr; R.verb_len = 0; R.cls = 0; R.bad = 1; R.chr = 0;
    uint32_t seq_bytes = 0;
    if (tid < nr) {
        *reinterpret_cast<uint4 *>(&R.rec) = reinterpret_cast<const uint4 *>(recs)[r];
        R.chr = chr_of[r];
        const uint32_t len = R.rec.len, pos = R.rec.pos;
        R.bad = (len == 0u || len > max_len || (fixed_len && len != fixed_len) || pos == 0u || R.chr >= g.n_chr ||
                 (uint64_t)(pos - 1u) > g.chr_len[R.chr] || (!R.rec.match && R.rec.n_ins > len)) ? 1u : 0u;
        if (R.bad) { dev_set_error(err, CBCG_ERR_CORRUPT, r); if (len == 0u || len > max_len) R.rec.len = 0; }
        seq_bytes = R.rec.len + 1u;
        if (cls) {
            const uint64_t ord = ids ? ids[r] : r;
            R.cls = cls[ord];
            if (R.cls >= 4u) {                            /* verbatim: its entry by binary search over the listed reads */
                uint64_t lo = 0, hi = n_exc;
                while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (exc_read[mid] < ord) lo = mid + 1; else hi = mid; }
                if (lo < n_exc && exc_read[lo] == ord && !R.bad &&
                    k6_cigar_ok(exc_text + exc_off[lo], (uint32_t)(exc_off[lo + 1] - exc_off[lo]), R.rec.len)) {
                    R.verb = exc_text + exc_off[lo]; R.verb_len = (uint32_t)(exc_off[lo + 1] - exc_off[lo]);
                } else if (!R.bad) dev_set_error(err, CBCG_ERR_FORMAT, r);
                R.cls = 0;
            }
        }
        S.len[tid] = (uint16_t)R.rec.len;
    }

    /* the tile's SEQ in K3's text */
    uint32_t incl = warp_incl_scan(seq_bytes);
    if (lane == 31u) S.warp_tot[warp] = incl;
    __syncthreads();
    uint32_t warp_base = 0, seq_total = 0;
#pragma unroll
    for (uint32_t k = 0; k < K6_TILE / 32u; k++) { const uint32_t t = S.warp_tot[k]; if (k < warp) warp_base += t; seq_total += t; }
    const uint32_t my_seq = warp_base + incl - seq_bytes;
    if (fixed_len) { if (tid == 0) S.seq_base = r0 * (uint64_t)(fixed_len + 1u); }
    else if (warp == 0) { const uint64_t b = lookback_exclusive(desc_seq, tile, seq_total, err); if (lane == 0) S.seq_base = b; }
    __syncthreads();
    const uint64_t seq_base = S.seq_base;
    const uint32_t head = (uint32_t)(seq_base & 15u);
    if (tid == 0) {
        const uint32_t bytes = (head + seq_total + 15u) & ~15u;
        mbar_expect_tx(&S.bar, bytes);
        tma_load_1d(s_seq, seq_text + (seq_base - head), bytes, &S.bar);
    }
    const uint8_t *my_seq_p = s_seq + head + my_seq;
    if (tid < nr) S.seq_src[tid] = head + my_seq;

    /* line sizes: the fast path needs no SEQ, so its reads are sized while the copy is in flight */
    uint32_t nm = 0, at_dummy = 0, line = 0;
    bool malformed = false;
    if (tid < nr && !R.verb) line = k6_line<false>(nullptr, R, edits, g, names, name_len, my_seq_p, false, &nm, &at_dummy, &malformed);
    mbar_wait(&S.bar, 0);
    if (tid < nr && R.verb) line = k6_line<false>(nullptr, R, edits, g, names, name_len, my_seq_p, false, &nm, &at_dummy, &malformed);
    if (malformed) dev_set_error(err, CBCG_ERR_CORRUPT, r);

    incl = warp_incl_scan(line);
    if (lane == 31u) S.warp_tot2[warp] = incl;
    __syncthreads();
    uint32_t tile_total = 0; warp_base = 0;
#pragma unroll
    for (uint32_t k = 0; k < K6_TILE / 32u; k++) { const uint32_t t = S.warp_tot2[k]; if (k < warp) warp_base += t; tile_total += t; }
    const uint32_t my_off = warp_base + incl - line;
    if (warp == 0) {
        const uint64_t b = lookback_exclusive(desc_out, tile, tile_total, err);
        if (lane == 0) { S.out_base = b; if (r0 + nr == n_reads) *total_bytes = b + tile_total; }
    }
    __syncthreads();
    const uint64_t out_base = S.out_base;
    if (out_base + tile_total > out_cap) { if (tid == 0) dev_set_error(err, CBCG_ERR_CAPACITY, r0); return; }
    uint8_t *gdst = out + out_base;

    const uint32_t shift = (uint32_t)((uint64_t)gdst & 15ull);
    if (shift + tile_total > img_cap) {                    /* CTA-uniform: lines too long for the image, straight to HBM */
        if (tid < nr) k6_line<true>(gdst + my_off, R, edits, g, names, name_len, my_seq_p, true, &nm, &at_dummy, &malformed);
        return;
    }
    uint8_t *img = s_img + shift;
    uint32_t seq_at = 0;
    if (tid < nr) {
        k6_line<true>(img + my_off, R, edits, g, names, name_len, my_seq_p, false, &nm, &seq_at, &malformed);
        S.line_off[tid] = my_off; S.seq_at[tid] = seq_at;
    }
    __syncthreads();
    /* SEQ fields, a warp per read: lanes on consecutive bytes */
    for (uint32_t i = warp; i < nr; i += K6_TILE / 32u) {
        const uint8_t *src = s_seq + S.seq_src[i];
        uint8_t *dst = img + S.line_off[i] + S.seq_at[i];
        const uint32_t len = S.len[i];
        for (uint32_t j = lane; j < len; j += 32u) dst[j] = src[j];
    }
    fence_proxy_async_smem();          /* generic-proxy smem writes -> visible to the bulk store */
    __syncthreads();
    const uint32_t h = min(tile_total, (16u - shift) & 15u);
    const uint32_t mid = (tile_total - h) & ~15u;
    const uint32_t tail = tile_total - h - mid;
    if (tid == 0 && mid) {
        tma_store_1d(gdst + h, img + h, mid);
        tma_store_commit_wait();
    }
    if (tid >= 32 && tid < 32 + h) gdst[tid - 32] = img[tid - 32];
    if (tid >= 64 && tid < 64 + tail) gdst[h + mid + (tid - 64)] = img[h + mid + (tid - 64)];
}

int launch_sam(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const uint16_t *edits, const DevGenome &g,
               const uint8_t *names, const uint32_t *name_len, const uint8_t *seq_text, uint32_t max_len, uint32_t fixed_len,
               const uint64_t *ids, const uint8_t *cls, const uint64_t *exc_read, const uint64_t *exc_off, const uint8_t *exc_text,
               uint64_t n_exc, uint8_t *out, uint64_t out_cap, uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_bytes,
               unsigned long long *err, cudaStream_t st) {
    if (!n_reads) return 0;
    if (max_len == 0 || max_len > CBCG_MAX_READ_LEN) return -1;
    const uint64_t tiles = sam_num_tiles(n_reads);
    const size_t smem = sizeof(K6Smem) + k6_stage_cap(max_len) + k6_img_cap(max_len) + 32u;
    const size_t smem_max = sizeof(K6Smem) + k6_stage_cap(CBCG_MAX_READ_LEN) + k6_img_cap(CBCG_MAX_READ_LEN) + 32u;
    if (cudaFuncSetAttribute(k6_sam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max) != cudaSuccess) return -1;
    if (cudaMemsetAsync(tile_desc, 0, 2u * tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
    k6_sam_kernel<<<(unsigned)tiles, K6_TILE, smem, st>>>(n_reads, recs, chr, edits, g, names, name_len, seq_text, max_len, fixed_len, ids, cls,
                                                          exc_read, exc_off, exc_text, n_exc, out, out_cap, tile_desc, tile_desc + tiles,
                                                          ticket, total_bytes, err);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
