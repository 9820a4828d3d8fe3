/*
 * k9_bam.cu -- K9: BAM records in BGZF blocks (cbcg_decode_bam).
 *
 * Runs after K3, over K3's text and the records the block decoder wrote (or K5 kept): the same reads, CIGAR, MD and NM as
 * K6's SAM lines (the field builders are sam_fields.cuh's), encoded as BAM (SAMv1 4.2) inside BGZF (SAMv1 4.1).
 *
 *   record: block_size, refID (the read's index in the header's name list: ref_id[genome ordinal]), pos = POS - 1,
 *     l_read_name 2, mapq 255, bin = reg2bin(pos, end) (end = pos + the CIGAR's M D N = X span, or pos + 1 when that is
 *     0), n_cigar_op, FLAG, l_seq, next_refID -1, next_pos -1, tlen 0, read_name "*\0", the CIGAR as u32 len << 4 | op
 *     (MIDNSHP=X), SEQ in the 4-bit code =ACMGRSVTWYHKDBN (high nibble first; any other byte is 15, N), QUAL l_seq x 0xff,
 *     then NM:C (NM:S above 255) and MD:Z. A record above K9_MAX_RECORD bytes is CBCG_ERR_FORMAT (the format's limits keep
 *     records under about 5.2 KB; only a pathological verbatim CIGAR reaches it), as is a verbatim operation longer than
 *     2^28 - 1.
 *   blocks: whole records; record i > 0 opens a block when floor(U_i / K9_BLOCK_CUT) != floor(U_{i-1} / K9_BLOCK_CUT),
 *     U_i the record bytes before it in the call. A block therefore holds fewer than K9_MAX_BLOCK = 57 344 bytes, and
 *     block q (q >= 1) starts at the first record with U_i >= q K9_BLOCK_CUT.
 *   deflate: one final fixed-Huffman block per BGZF block. Every record byte is a literal except QUAL's: one literal 0xff,
 *     then one match <l_seq - 1, distance 1> when l_seq - 1 >= 3 (else literals). End-of-block, zero bits to the byte.
 *     Worst case 57 343 nine-bit literals: 64 539 bytes of BGZF block, under the 65 536 limit.
 *
 * B200 design.
 *   k9_bam_record_kernel: K6's shape. One CTA per tile of K9_TILE reads, a thread per read; the tile's SEQ is staged from
 *     K3's text by one TMA bulk copy; a counting pass sizes each record, a CTA scan and a decoupled look-back (tile order
 *     from an atomic ticket) give its offset in the uncompressed stream; records are written into a shared-memory image
 *     that leaves by one TMA bulk store (plus byte stores for the ragged ends), straight to HBM when a tile's records do
 *     not fit it. Each record's offset goes to rec_off; the record that ends where the next one opens a block writes that
 *     block's first record to block_first, and the last record writes the totals.
 *   k9_bgzf_kernel: one CTA of K9_BGZF_THREADS per BGZF block (tile order from an atomic ticket). The block's records come
 *     in by one TMA bulk copy. Each thread takes a contiguous chunk of the block's bytes: a pass computes the chunk's raw
 *     CRC32 and its deflate bit cost (8 or 9 bits per literal, the QUAL match's code and extra bits on the byte after the
 *     first 0xff, 0 on the rest of the run); the chunk CRCs are combined by GF(2) shifts (zlib's crc32_combine, bgzf.cuh), a CTA scan
 *     of the costs gives each chunk's bit offset, and a second pass writes the codes into a zeroed shared-memory bit image
 *     (shared atomicOr on the words a chunk shares with its neighbours). A decoupled look-back over the block sizes gives
 *     its output offset; the block leaves by 16-byte vector stores.
 */
#include "common.cuh"
#include "internal.h"
#include "sam_fields.cuh"
#include "bgzf.cuh"

#define K9_TILE 128u
#define K9_MAX_RECORD 8192u
#define K9_MAX_BLOCK (K9_BLOCK_CUT + K9_MAX_RECORD)
#define K9_BGZF_THREADS 1024u
#define K9_MIN_RECORD 49u                                   /* 36 fixed + "*\0" + 1 SEQ + 1 QUAL + NM:C + "MD" 'Z' "0\0" */
#define K9_MAX_RECS (K9_MAX_BLOCK / K9_MIN_RECORD + 2u)
#define K9_STAGE_BYTES (K9_MAX_BLOCK + 32u)
#define K9_IMG_BYTES (20u + 64516u + 8u + 16u)              /* 2 pad + 18 header, deflate bytes (<= 64 514), footer, slack */

uint64_t bam_num_tiles(uint64_t n_reads) { return (n_reads + K9_TILE - 1u) / K9_TILE; }

/* ---------------------------------------------------------------- records */
/* image bytes per read of the tile: room for an ordinary record (SEQ and QUAL take 3 / 2 per base); a tile that needs more
   writes straight to HBM */
static inline CBCG_HD uint32_t k9_img_cap(uint32_t max_len) { return K9_TILE * ((3u * max_len) / 2u + 96u); }
static inline CBCG_HD uint32_t k9_stage_cap(uint32_t max_len) { return ((K9_TILE * (max_len + 1u) + 32u + 15u) & ~15u); }

__device__ __forceinline__ void st_le16(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
__device__ __forceinline__ void st_le32(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }

/* BAM CIGAR: counts the operations and the reference span, and writes them (W) as u32 len << 4 | op. */
template <bool W> struct K9Cig {
    uint8_t *p; uint32_t n, span; bool too_long;
    __device__ __forceinline__ void cig(uint32_t cnt, uint32_t op) {
        const uint32_t code = op == 'M' ? 0u : op == 'I' ? 1u : op == 'D' ? 2u : op == 'N' ? 3u : op == 'S' ? 4u : op == 'H' ? 5u
                            : op == 'P' ? 6u : op == '=' ? 7u : 8u;
        if (cnt >= (1u << 28)) too_long = true;
        if (W) st_le32(p + 4u * n, (cnt << 4) | code);
        if (code == 0u || code == 2u || code == 3u || code == 7u || code == 8u) span += cnt;
        n++;
    }
};

/* the spec's reg2bin over [beg, end) */
__device__ __forceinline__ uint32_t k9_reg2bin(int32_t beg, int32_t end) {
    --end;
    if (beg >> 14 == end >> 14) return ((1u << 15) - 1u) / 7u + (uint32_t)(beg >> 14);
    if (beg >> 17 == end >> 17) return ((1u << 12) - 1u) / 7u + (uint32_t)(beg >> 17);
    if (beg >> 20 == end >> 20) return ((1u << 9) - 1u) / 7u + (uint32_t)(beg >> 20);
    if (beg >> 23 == end >> 23) return ((1u << 6) - 1u) / 7u + (uint32_t)(beg >> 23);
    if (beg >> 26 == end >> 26) return ((1u << 3) - 1u) / 7u + (uint32_t)(beg >> 26);
    return 0u;
}

/* htslib's seq_nt16_table: =ACMGRSVTWYHKDBN in either case, anything else 15 */
__device__ __forceinline__ uint32_t k9_nt16(uint32_t c) {
    if (c >= 'a' && c <= 'z') c -= 32u;
    switch (c) {
    case '=': return 0u;  case 'A': return 1u;  case 'C': return 2u;  case 'M': return 3u;
    case 'G': return 4u;  case 'R': return 5u;  case 'S': return 6u;  case 'V': return 7u;
    case 'T': return 8u;  case 'W': return 9u;  case 'Y': return 10u; case 'H': return 11u;
    case 'K': return 12u; case 'D': return 13u; case 'B': return 14u; default: return 15u;
    }
}

struct K9Read {
    cbcg_read_rec rec;
    uint32_t chr, cls, bad;
    int32_t ref_id;
    const uint8_t *verb; uint32_t verb_len;            /* class 4 with a valid text */
};

/* What the counting pass learns and the writing pass uses. */
struct K9Fields { uint32_t n_ops, span, nm, md_len, ins_bases; bool malformed, too_long; };

template <bool W> __device__ static void k9_cigar(K9Cig<W> &c, const K9Read &R, const uint16_t *e, uint32_t nd, uint32_t ns, uint32_t ni,
                                                  uint32_t *ins_bases) {
    if (R.bad) return;
    if (R.verb) {                                       /* passed k6_cigar_ok: digits then one of MIDSHP=X, to the end */
        uint32_t i = 0;
        while (i < R.verb_len) {
            uint32_t num = 0;
            while (R.verb[i] >= '0' && R.verb[i] <= '9') num = num * 10u + (uint32_t)(R.verb[i++] - '0');
            c.cig(num, R.verb[i++]);
        }
    } else *ins_bases = k6_cigar_implied(c, R.rec.len, nd, ni, e, e + nd + ns, R.cls);
}

/* Counting pass: the fields' sizes and NM (as K6's line: MD from the record's edits or the verbatim CIGAR's walk). */
__device__ static uint32_t k9_count(K9Fields &F, const K9Read &R, const uint16_t *edits, const DevGenome &g, const uint8_t *seq) {
    const cbcg_read_rec &r = R.rec;
    const uint32_t len = r.len;
    const uint32_t nd = r.match ? 0u : r.n_dels, ns = r.match ? 0u : r.n_snps, ni = r.match ? 0u : r.n_ins;
    const uint16_t *e = edits + r.edit_off;
    const uint8_t *ref = R.bad ? nullptr : g.bases + g.chr_off[R.chr] + (r.pos - 1u);
    K9Cig<false> c{ nullptr, 0u, 0u, false };
    F.ins_bases = 0; F.malformed = false;
    k9_cigar(c, R, e, nd, ns, ni, &F.ins_bases);
    F.n_ops = c.n; F.span = c.span; F.too_long = c.too_long;
    K6Out<false> md{ nullptr, 0u };
    if (R.bad) { F.nm = 0; md.put('0'); }
    else if (R.verb) k6_md_walk(md, R.verb, R.verb_len, seq, ref, &F.nm);
    else F.nm = k6_md_edits(md, len - ni, nd, ns, e, e + nd, ref, &F.malformed) + F.ins_bases + nd;
    F.md_len = md.n;
    return 36u + 2u + 4u * F.n_ops + (len + 1u) / 2u + len + (F.nm <= 255u ? 4u : 5u) + 3u + F.md_len + 1u;
}

/* Writing pass: the record of `size` bytes at dst. */
__device__ static void k9_write(uint8_t *dst, uint32_t size, const K9Fields &F, const K9Read &R, const uint16_t *edits, const DevGenome &g,
                                const uint8_t *seq) {
    const cbcg_read_rec &r = R.rec;
    const uint32_t len = r.len;
    const uint32_t nd = r.match ? 0u : r.n_dels, ns = r.match ? 0u : r.n_snps, ni = r.match ? 0u : r.n_ins;
    const uint16_t *e = edits + r.edit_off;
    const uint8_t *ref = R.bad ? nullptr : g.bases + g.chr_off[R.chr] + (r.pos - 1u);
    const int32_t beg = (int32_t)r.pos - 1;
    st_le32(dst, size - 4u);
    st_le32(dst + 4, (uint32_t)(R.bad ? -1 : R.ref_id));
    st_le32(dst + 8, (uint32_t)beg);
    dst[12] = 2u; dst[13] = 255u;
    st_le16(dst + 14, k9_reg2bin(beg, beg + (int32_t)(F.span ? F.span : 1u)));
    st_le16(dst + 16, F.n_ops);
    st_le16(dst + 18, r.flag);
    st_le32(dst + 20, len);
    st_le32(dst + 24, 0xffffffffu); st_le32(dst + 28, 0xffffffffu); st_le32(dst + 32, 0u);
    dst[36] = '*'; dst[37] = 0u;
    K9Cig<true> c{ dst + 38, 0u, 0u, false };
    uint32_t ins_dummy = 0;
    k9_cigar(c, R, e, nd, ns, ni, &ins_dummy);
    uint8_t *s = dst + 38u + 4u * F.n_ops;
    for (uint32_t j = 0; j < len; j += 2u)
        s[j >> 1] = (uint8_t)((k9_nt16(seq[j]) << 4) | (j + 1u < len ? k9_nt16(seq[j + 1u]) : 0u));
    uint8_t *q = s + (len + 1u) / 2u;
    for (uint32_t j = 0; j < len; j++) q[j] = 0xffu;
    uint8_t *t = q + len;
    t[0] = 'N'; t[1] = 'M';
    if (F.nm <= 255u) { t[2] = 'C'; t[3] = (uint8_t)F.nm; t += 4; }
    else { t[2] = 'S'; st_le16(t + 3, F.nm); t += 5; }
    t[0] = 'M'; t[1] = 'D'; t[2] = 'Z';
    K6Out<true> md{ t + 3, 0u };
    bool malformed = false;
    if (R.bad) md.put('0');
    else if (R.verb) { uint32_t dummy; k6_md_walk(md, R.verb, R.verb_len, seq, ref, &dummy); }
    else k6_md_edits(md, len - ni, nd, ns, e, e + nd, ref, &malformed);
    md.put(0u);
}

struct K9Smem {
    uint64_t bar;
    uint64_t seq_base, out_base;
    uint32_t tile;
    uint32_t warp_tot[K9_TILE / 32u], warp_tot2[K9_TILE / 32u];
    __align__(16) uint8_t dyn[16];    /* stage (k9_stage_cap), then the image (k9_img_cap + 32): dynamic */
};

__global__ void __launch_bounds__(K9_TILE)
k9_bam_record_kernel(uint64_t n_reads, const cbcg_read_rec *__restrict__ recs, const uint32_t *__restrict__ chr_of, const uint16_t *__restrict__ edits,
                     DevGenome g, const int32_t *__restrict__ ref_id, const uint8_t *__restrict__ seq_text, uint32_t max_len, uint32_t fixed_len,
                     const uint64_t *__restrict__ ids, const uint8_t *__restrict__ cls, const uint64_t *__restrict__ exc_read,
                     const uint64_t *__restrict__ exc_off, const uint8_t *__restrict__ exc_text, uint64_t n_exc, uint8_t *__restrict__ out,
                     uint64_t out_cap, uint64_t *__restrict__ rec_off, uint32_t *__restrict__ block_first, uint64_t *desc_seq, uint64_t *desc_out,
                     uint32_t *ticket, uint64_t *totals, unsigned long long *err) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    K9Smem &S = *reinterpret_cast<K9Smem *>(smem_raw);
    uint8_t *const s_seq = S.dyn, *const s_img = S.dyn + k9_stage_cap(max_len);
    const uint32_t img_cap = k9_img_cap(max_len);
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) {
        S.tile = atomicAdd(ticket, 1u);
        mbar_init(&S.bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    const uint32_t tile = S.tile;
    const uint64_t r0 = (uint64_t)tile * K9_TILE, r = r0 + tid;
    const uint32_t nr = (uint32_t)min((uint64_t)K9_TILE, n_reads - r0);

    K9Read R;
    R.verb = nullptr; R.verb_len = 0; R.cls = 0; R.bad = 1; R.chr = 0; R.ref_id = -1;
    uint32_t seq_bytes = 0;
    if (tid < nr) {
        *reinterpret_cast<uint4 *>(&R.rec) = reinterpret_cast<const uint4 *>(recs)[r];
        R.chr = chr_of[r];
        const uint32_t len = R.rec.len, pos = R.rec.pos;
        R.bad = (len == 0u || len > max_len || (fixed_len && len != fixed_len) || pos == 0u || R.chr >= g.n_chr ||
                 (uint64_t)(pos - 1u) > g.chr_len[R.chr] || (!R.rec.match && R.rec.n_ins > len) || ref_id[R.chr] < 0) ? 1u : 0u;
        if (R.bad) { dev_set_error(err, CBCG_ERR_CORRUPT, r); if (len == 0u || len > max_len) R.rec.len = 0; }
        else R.ref_id = ref_id[R.chr];
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
    }

    /* the tile's SEQ in K3's text */
    uint32_t incl = warp_incl_scan(seq_bytes);
    if (lane == 31u) S.warp_tot[warp] = incl;
    __syncthreads();
    uint32_t warp_base = 0, seq_total = 0;
#pragma unroll
    for (uint32_t k = 0; k < K9_TILE / 32u; k++) { const uint32_t t = S.warp_tot[k]; if (k < warp) warp_base += t; seq_total += t; }
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

    /* record sizes: the fast path needs no SEQ, so its reads are sized while the copy is in flight */
    K9Fields F{};
    uint32_t size = 0;
    if (tid < nr && !R.verb) size = k9_count(F, R, edits, g, my_seq_p);
    mbar_wait(&S.bar, 0);
    if (tid < nr && R.verb) size = k9_count(F, R, edits, g, my_seq_p);
    if (F.malformed) dev_set_error(err, CBCG_ERR_CORRUPT, r);
    if (tid < nr && (size > K9_MAX_RECORD || F.too_long)) dev_set_error(err, CBCG_ERR_FORMAT, r);

    incl = warp_incl_scan(size);
    if (lane == 31u) S.warp_tot2[warp] = incl;
    __syncthreads();
    uint32_t tile_total = 0; warp_base = 0;
#pragma unroll
    for (uint32_t k = 0; k < K9_TILE / 32u; k++) { const uint32_t t = S.warp_tot2[k]; if (k < warp) warp_base += t; tile_total += t; }
    const uint32_t my_off = warp_base + incl - size;
    if (warp == 0) {
        const uint64_t b = lookback_exclusive(desc_out, tile, tile_total, err);
        if (lane == 0) S.out_base = b;
    }
    __syncthreads();
    const uint64_t out_base = S.out_base;
    if (out_base + tile_total > out_cap) { if (tid == 0) dev_set_error(err, CBCG_ERR_INTERNAL, r0); return; }
    if (tid < nr) {                                        /* offsets, block starts and, from the last record, the totals */
        const uint64_t u = out_base + my_off, end = u + size;
        rec_off[r] = u;
        if (r == 0) block_first[0] = 0;
        if (r + 1 < n_reads) { if (u / K9_BLOCK_CUT != end / K9_BLOCK_CUT) block_first[end / K9_BLOCK_CUT] = (uint32_t)(r + 1); }
        else {
            const uint64_t nb = u / K9_BLOCK_CUT + 1u;
            rec_off[n_reads] = end; block_first[nb] = (uint32_t)n_reads;
            totals[0] = end; totals[1] = nb;
        }
    }
    uint8_t *gdst = out + out_base;
    const uint32_t shift = (uint32_t)((uint64_t)gdst & 15ull);
    if (shift + tile_total > img_cap) {                    /* CTA-uniform: records too long for the image, straight to HBM */
        if (tid < nr) k9_write(gdst + my_off, size, F, R, edits, g, my_seq_p);
        return;
    }
    uint8_t *img = s_img + shift;
    if (tid < nr) k9_write(img + my_off, size, F, R, edits, g, my_seq_p);
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

/* ---------------------------------------------------------------- BGZF blocks */
/* A length symbol of the fixed code: its code reversed for LSB-first output, the code's bits, extra bits and their value. */
__device__ __forceinline__ void k9_len_sym(uint32_t L, uint32_t &code, uint32_t &nb, uint32_t &eb, uint32_t &ev) {
    uint32_t sym;
    if (L <= 10u) { sym = 254u + L; eb = 0; ev = 0; }
    else if (L == 258u) { sym = 285u; eb = 0; ev = 0; }
    else { eb = 29u - __clz(L - 3u); sym = 257u + 4u * eb + ((L - 3u) >> eb); ev = (L - 3u) & ((1u << eb) - 1u); }
    if (sym < 280u) { code = __brev(sym - 256u) >> 25; nb = 7u; }
    else { code = __brev(0xc0u + sym - 280u) >> 24; nb = 8u; }
}
__device__ __forceinline__ uint32_t k9_lit_bits(uint32_t v) { return v < 144u ? 8u : 9u; }
__device__ __forceinline__ uint32_t k9_lit_code(uint32_t v) { return v < 144u ? __brev(0x30u + v) >> 24 : __brev(0x190u + v - 144u) >> 23; }

/* LSB-first bit writer into the zeroed shared image: the first word it flushes and its last partial word may be shared
   with the neighbouring chunks (atomicOr); the words in between are its own. */
struct K9Bits {
    uint32_t *img; uint32_t word; uint64_t acc; uint32_t n; bool first;
    __device__ __forceinline__ void put(uint32_t v, uint32_t nb) {
        acc |= (uint64_t)v << n; n += nb;
        if (n >= 32u) {
            if (first) { atomicOr(&img[word], (uint32_t)acc); first = false; } else img[word] = (uint32_t)acc;
            word++; acc >>= 32; n -= 32u;
        }
    }
    __device__ __forceinline__ void finish() { if (n) atomicOr(&img[word], (uint32_t)acc); }
};

struct K9bSmem {
    uint64_t bar;
    uint64_t in_base, out_base;
    uint32_t tile, first, nrec, bytes, bad;
    uint32_t warp_bits[K9_BGZF_THREADS / 32u], warp_crc[K9_BGZF_THREADS / 32u];
    uint32_t crc_tab[256];
    uint16_t rs[K9_MAX_RECS + 1u];                        /* each record's start in the block, then the block's size */
    __align__(16) uint8_t dyn[16];                        /* stage (K9_STAGE_BYTES), then the block image (K9_IMG_BYTES): dynamic */
};

/* the record of the block that holds byte p: the last k with rs[k] <= p */
__device__ __forceinline__ uint32_t k9_find(const uint16_t *rs, uint32_t nrec, uint32_t p) {
    uint32_t lo = 0, hi = nrec;                           /* rs[lo] <= p < rs[hi] */
    while (hi - lo > 1u) { const uint32_t mid = (lo + hi) >> 1; if (rs[mid] <= p) lo = mid; else hi = mid; }
    return lo;
}
/* QUAL of record k: its first byte and l_seq (l_read_name is 2) */
__device__ __forceinline__ void k9_qual(const uint8_t *raw, const uint16_t *rs, uint32_t k, uint32_t &qa, uint32_t &ql) {
    const uint8_t *p = raw + rs[k];
    const uint32_t n_ops = p[16] | (uint32_t)p[17] << 8, l_seq = p[20] | (uint32_t)p[21] << 8 | (uint32_t)p[22] << 16 | (uint32_t)p[23] << 24;
    ql = l_seq; qa = rs[k] + 38u + 4u * n_ops + (l_seq + 1u) / 2u;
}

__global__ void __launch_bounds__(K9_BGZF_THREADS)
k9_bgzf_kernel(const uint8_t *__restrict__ stream, const uint64_t *__restrict__ rec_off, const uint32_t *__restrict__ block_first,
               uint32_t n_blocks, uint8_t *__restrict__ out, uint64_t *desc, uint32_t *ticket, uint64_t *total_bytes, unsigned long long *err) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    K9bSmem &S = *reinterpret_cast<K9bSmem *>(smem_raw);
    uint8_t *const stage = S.dyn, *const blk = S.dyn + K9_STAGE_BYTES;
    uint32_t *const words = reinterpret_cast<uint32_t *>(blk + 20);   /* the deflate data, after 2 pad + 18 header bytes */
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) {
        const uint32_t q = atomicAdd(ticket, 1u);
        S.tile = q;
        const uint32_t f = block_first[q], l = block_first[q + 1u];
        const uint64_t a = rec_off[f], b = rec_off[l];
        S.first = f; S.nrec = l - f; S.in_base = a;
        S.bad = (l <= f || l - f > K9_MAX_RECS || b - a > K9_MAX_BLOCK) ? 1u : 0u;
        S.bytes = S.bad ? 0u : (uint32_t)(b - a);
        if (S.bad) dev_set_error(err, CBCG_ERR_FORMAT, f);
        mbar_init(&S.bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    const uint32_t B = S.bytes, nrec = S.nrec;
    const uint32_t head = (uint32_t)(S.in_base & 15u);
    if (tid == 0 && B) {
        const uint32_t bytes = (head + B + 15u) & ~15u;
        mbar_expect_tx(&S.bar, bytes);
        tma_load_1d(stage, stream + (S.in_base - head), bytes, &S.bar);
    }
    for (uint32_t k = tid; k < 256u; k += K9_BGZF_THREADS) {
        S.crc_tab[k] = bgzf_crc_table_entry(k);
    }
    if (B) for (uint32_t k = tid; k <= nrec; k += K9_BGZF_THREADS) S.rs[k] = (uint16_t)(rec_off[S.first + k] - S.in_base);
    for (uint32_t k = tid; k < K9_IMG_BYTES / 4u; k += K9_BGZF_THREADS) reinterpret_cast<uint32_t *>(blk)[k] = 0u;
    if (B) mbar_wait(&S.bar, 0);
    __syncthreads();
    const uint8_t *raw = stage + head;

    /* pass 1: the chunk's raw CRC and bit cost */
    const uint32_t ch = (B + K9_BGZF_THREADS - 1u) / K9_BGZF_THREADS;
    const uint32_t a = min(B, tid * ch), b = min(B, a + ch);
    uint32_t crc = 0, bits = 0;
    uint32_t k = 0, qa = 0, ql = 0, next = 0;
    if (a < b) { k = k9_find(S.rs, nrec, a); k9_qual(raw, S.rs, k, qa, ql); next = S.rs[k + 1u]; }
    for (uint32_t p = a; p < b; p++) {
        while (p >= next) { k++; k9_qual(raw, S.rs, k, qa, ql); next = S.rs[k + 1u]; }
        const uint32_t v = raw[p];
        crc = S.crc_tab[(crc ^ v) & 0xffu] ^ (crc >> 8);
        if (ql >= 4u && p > qa && p < qa + ql) {
            if (p == qa + 1u) { uint32_t code, nb, eb, ev; k9_len_sym(ql - 1u, code, nb, eb, ev); bits += nb + eb + 5u; }
        } else bits += k9_lit_bits(v);
    }
    /* the block's CRC: each chunk's raw CRC shifted past the bytes after it, the initial value's shifted past the block */
    uint32_t part = a < b ? bgzf_crc_shift(crc, B - b) : 0u;
    for (int o = 16; o > 0; o >>= 1) part ^= __shfl_xor_sync(FULL_MASK, part, o);
    const uint32_t incl = warp_incl_scan(bits);
    if (lane == 31u) { S.warp_bits[warp] = incl; S.warp_crc[warp] = part; }
    __syncthreads();
    uint32_t warp_base = 0, total_bits = 0, crc_all = 0;
    for (uint32_t w = 0; w < K9_BGZF_THREADS / 32u; w++) {
        const uint32_t t = S.warp_bits[w];
        if (w < warp) warp_base += t;
        total_bits += t; crc_all ^= S.warp_crc[w];
    }
    /* pass 2: the codes, after BFINAL 1 and BTYPE 01 */
    K9Bits W{ words, 0u, 0ull, 0u, true };
    const uint32_t at = 3u + warp_base + incl - bits;
    W.word = at >> 5; W.n = at & 31u;
    if (a < b) { k = k9_find(S.rs, nrec, a); k9_qual(raw, S.rs, k, qa, ql); next = S.rs[k + 1u]; }
    for (uint32_t p = a; p < b; p++) {
        while (p >= next) { k++; k9_qual(raw, S.rs, k, qa, ql); next = S.rs[k + 1u]; }
        const uint32_t v = raw[p];
        if (ql >= 4u && p > qa && p < qa + ql) {
            if (p == qa + 1u) {
                uint32_t code, nb, eb, ev;
                k9_len_sym(ql - 1u, code, nb, eb, ev);
                W.put(code, nb);
                if (eb) W.put(ev, eb);
                W.put(0u, 5u);                            /* distance 1: distance code 0, five zero bits */
            }
        } else W.put(k9_lit_code(v), k9_lit_bits(v));
    }
    W.finish();
    if (tid == 0) atomicOr(&words[0], 3u);
    /* end-of-block (seven zero bits), then zero bits to the byte */
    const uint32_t dbytes = (3u + total_bits + 7u + 7u) / 8u;
    const uint32_t size = B ? 18u + dbytes + 8u : 0u;
    if (warp == 0) {
        const uint64_t o = lookback_exclusive(desc, S.tile, size, err);
        if (lane == 0) { S.out_base = o; if (S.tile + 1u == n_blocks) *total_bytes = o + size; }
    }
    __syncthreads();
    if (!size) return;
    if (tid == 0) {
        const uint8_t h18[18] = { 0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, (uint8_t)(size - 1u), (uint8_t)((size - 1u) >> 8) };
        for (int j = 0; j < 18; j++) blk[2 + j] = h18[j];
        const uint32_t crc32 = bgzf_crc_finish(crc_all, B);
        uint8_t *f = blk + 20 + dbytes;
        st_le32(f, crc32); st_le32(f + 4, B);
    }
    __syncthreads();
    /* the block [2, 2 + size) of the image -> out: byte stores to 16-byte alignment, 16-byte vector stores, byte stores */
    uint8_t *gdst = out + S.out_base;
    const uint32_t h = min(size, (uint32_t)((16u - ((uint64_t)gdst & 15u)) & 15u));
    const uint32_t mid = (size - h) & ~15u;
    const uint32_t tail = size - h - mid;
    if (tid < h) gdst[tid] = blk[2 + tid];
    for (uint32_t j = h + 16u * tid; j < h + mid; j += 16u * K9_BGZF_THREADS) {
        uint4 v;
        v.x = lds_u32_unaligned(blk, 2 + j); v.y = lds_u32_unaligned(blk, 6 + j);
        v.z = lds_u32_unaligned(blk, 10 + j); v.w = lds_u32_unaligned(blk, 14 + j);
        *reinterpret_cast<uint4 *>(gdst + j) = v;
    }
    if (tid >= 32u && tid < 32u + tail) gdst[h + mid + (tid - 32u)] = blk[2 + h + mid + (tid - 32u)];
}

int launch_bam_records(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const uint16_t *edits, const DevGenome &g,
                       const int32_t *ref_id, const uint8_t *seq_text, uint32_t max_len, uint32_t fixed_len, const uint64_t *ids,
                       const uint8_t *cls, const uint64_t *exc_read, const uint64_t *exc_off, const uint8_t *exc_text, uint64_t n_exc,
                       uint8_t *stream, uint64_t stream_cap, uint64_t *rec_off, uint32_t *block_first, uint64_t *tile_desc, uint32_t *ticket,
                       uint64_t *totals, unsigned long long *err, cudaStream_t st) {
    if (!n_reads) return 0;
    if (max_len == 0 || max_len > CBCG_MAX_READ_LEN) return -1;
    const uint64_t tiles = bam_num_tiles(n_reads);
    const size_t smem = sizeof(K9Smem) + k9_stage_cap(max_len) + k9_img_cap(max_len) + 32u;
    const size_t smem_max = sizeof(K9Smem) + k9_stage_cap(CBCG_MAX_READ_LEN) + k9_img_cap(CBCG_MAX_READ_LEN) + 32u;
    if (cudaFuncSetAttribute(k9_bam_record_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max) != cudaSuccess) return -1;
    if (cudaMemsetAsync(tile_desc, 0, 2u * tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
    k9_bam_record_kernel<<<(unsigned)tiles, K9_TILE, smem, st>>>(n_reads, recs, chr, edits, g, ref_id, seq_text, max_len, fixed_len, ids, cls,
                                                                 exc_read, exc_off, exc_text, n_exc, stream, stream_cap, rec_off, block_first,
                                                                 tile_desc, tile_desc + tiles, ticket, totals, err);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_bgzf(const uint8_t *stream, const uint64_t *rec_off, const uint32_t *block_first, uint32_t n_blocks, uint8_t *out,
                uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_bytes, unsigned long long *err, cudaStream_t st) {
    if (!n_blocks) return 0;
    const size_t smem = sizeof(K9bSmem) + K9_STAGE_BYTES + K9_IMG_BYTES;
    if (cudaFuncSetAttribute(k9_bgzf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaMemsetAsync(tile_desc, 0, n_blocks * sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
    k9_bgzf_kernel<<<n_blocks, K9_BGZF_THREADS, smem, st>>>(stream, rec_off, block_first, n_blocks, out, tile_desc, ticket, total_bytes, err);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
