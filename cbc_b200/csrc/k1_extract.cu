/*
 * k1_extract.cu -- K1: per-read edit extraction (hot path part 1).
 *
 * Replaces compress_edits + add_snps_to_array of the reference (src/read_compression.c:265-606,
 * 613-701) minus the symbol emission: for every read it decides the perfect-match bit
 * (:291-296) and, for the others, walks CIGAR and MD into the deletion / SNP / insertion
 * position-delta lists the reference's coder consumes (:308-552).
 *
 * B200 design. One CTA per tile of K1_TILE position-adjacent reads:
 *   - the tile's SEQ bytes (contiguous in the pool) and the reference window under its first reads
 *     are staged into shared memory by two 1-D TMA bulk copies completing on one mbarrier;
 *   - phase 1, warp per read: 32-bit word compare of SEQ against the window (ballot -> match bit);
 *   - phase 2, lane per read: serial CIGAR/MD walk of the non-matching reads, counting edits;
 *   - a CTA scan of the counts and a decoupled look-back across tiles give every read its slot in
 *     the edit array in ONE pass over the input (no count kernel + scan kernel + write kernel);
 *   - phase 3, lane per read: the same walk again, now writing u16 edit entries and the 16-byte record.
 * Algorithmic HBM bytes per read: L + CIGAR + MD + 24 (fixed fields) + L/coverage (window) + 16 + 2*edits.
 */
#include <algorithm>
#include "common.cuh"
#include "internal.h"

#define K1_TILE     128u          /* reads per tile == threads per CTA */
#define K1_WARPS    (K1_TILE / 32u)
#define K1_REF_CAP  8192u         /* most bytes of reference window staged per tile (DevBatch.ref_cap picks less for dense batches) */

uint64_t extract_num_tiles(uint64_t n_reads) { return (n_reads + K1_TILE - 1) / K1_TILE; }

/* ------------------------------------------------------------------------------------------------
 * The resumable MD walker: add_snps_to_array (src/read_compression.c:613-701) and
 * compute_num_digits (:720-743). State (ptr, cum) mirrors the reference's statics prevEditPtr / cumPos. */
struct MdWalk {
    const uint8_t *md;
    uint32_t n, ptr, cum;
    __device__ __forceinline__ uint32_t ch(uint32_t off) const { return off < n ? md[off] : 0u; }
    __device__ __forceinline__ uint32_t atoi_at(uint32_t off) const {
        uint32_t v = 0;
        while (off < n) {
            uint32_t c = md[off];
            if (c < '0' || c > '9') break;
            v = v * 10u + (c - '0');
            off++;
        }
        return v;
    }
};
__device__ __forceinline__ uint32_t num_digits(uint32_t x) {
    uint32_t d = 1;
    while (x >= 10u && d < 9u) { x /= 10u; d++; }
    return d;
}
__device__ __forceinline__ bool is_digit(uint32_t c) { return c >= '0' && c <= '9'; }

#define K1_ECACHE 4u          /* edits per read remembered from the count pass (kind in bits 14..15) */
struct EditSink {
    uint16_t *dst;          /* NULL: count only */
    uint32_t nd_total, ns_total;   /* write mode: counts from the count pass (slot bases) */
    uint32_t n_dels, n_snps, n_ins;
    int err;
    uint16_t *cache;        /* count pass: first K1_ECACHE entries in emission order (shared memory), or NULL */
    __device__ __forceinline__ void remember(uint32_t kind, uint32_t e) {
        const uint32_t k = n_dels + n_snps + n_ins;
        if (cache && k < K1_ECACHE) cache[k] = (uint16_t)(e | (kind << 14));
    }
    __device__ __forceinline__ void del(uint32_t delta) {
        if (delta > 255u) err = 1;
        if (dst && n_dels < 255u) dst[n_dels] = CBCG_EDIT(delta & 0xffu, 0, 0);
        remember(0u, CBCG_EDIT(delta & 0xffu, 0, 0));
        n_dels++;
    }
    __device__ __forceinline__ void snp(uint32_t delta, uint32_t target, uint32_t refb) {
        if (delta > 255u) err = 1;
        if (dst && n_snps < 255u) dst[nd_total + n_snps] = CBCG_EDIT(delta & 0xffu, target, refb);
        remember(1u, CBCG_EDIT(delta & 0xffu, target, refb));
        n_snps++;
    }
    __device__ __forceinline__ void ins(uint32_t delta, uint32_t target) {
        if (delta > 255u) err = 1;
        if (dst && n_ins < 255u) dst[nd_total + ns_total + n_ins] = CBCG_EDIT(delta & 0xffu, target, CBCG_BP_O);
        remember(2u, CBCG_EDIT(delta & 0xffu, target, CBCG_BP_O));
        n_ins++;
    }
};

/* Returns non-zero while SNPs may remain, 0 when the MD string is used up. */
__device__ static int md_walk(MdWalk &w, EditSink &out, uint32_t insertion_pos, const uint8_t *read, uint32_t read_len) {
    while (w.ch(w.ptr) != 0) {
        /* look ahead: matches up to the next mismatch, across deletions (:626-649) */
        uint32_t pos = w.atoi_at(w.ptr), temp = pos;
        uint32_t o = w.ptr + num_digits(pos);
        uint32_t c = w.ch(o); o++;
        bool hit_end = false;
        while (c == '^') {
            while (w.ch(o) != 0 && !is_digit(w.ch(o))) o++;
            uint32_t v = w.atoi_at(o);
            temp += v; o += num_digits(v);
            c = w.ch(o); o++;
            if (c == 0) { hit_end = true; break; }
        }
        if (hit_end) break;
        if (w.cum + temp >= insertion_pos) { w.cum++; return 1; }          /* :656-659 */
        /* consume (:661-682) */
        w.ptr += num_digits(pos);
        c = w.ch(w.ptr); w.ptr++;
        while (c == '^') {
            while (w.ch(w.ptr) != 0 && !is_digit(w.ch(w.ptr))) w.ptr++;
            uint32_t v = w.atoi_at(w.ptr);
            pos += v; w.ptr += num_digits(v);
            c = w.ch(w.ptr); w.ptr++;
        }
        if (c == 0) break;
        w.cum += pos;
        out.snp(pos, base_code(w.cum < read_len ? read[w.cum] : 0u), base_code(c));
        w.cum++;
        if (w.ch(w.ptr) == 0) break;
        if (out.n_snps > 1024u) { out.err = 1; break; }
    }
    w.ptr = 0; w.cum = 0;
    return 0;
}

/* CIGAR walk of compress_edits (src/read_compression.c:308-552). read points into shared memory. */
__device__ static void walk_read(const uint8_t *read, uint32_t len, const uint8_t *cigar, uint32_t cigar_len,
                                 const uint8_t *md, uint32_t md_len, EditSink &out) {
    MdWalk w = { md, md_len, 0u, 0u };
    uint32_t M = 0, prev_i = 0, prev_d = 0;
    int last_snp = 1, first = 1;
    uint32_t i = 0;
    while (i < cigar_len) {
        uint32_t num = 0, j = i;
        while (j < cigar_len && is_digit(cigar[j])) num = num * 10u + (uint32_t)(cigar[j++] - '0');
        if (j >= cigar_len) { out.err = 1; return; }
        uint32_t op = cigar[j];
        if (num > 1024u && op != 'H' && op != 'P') { out.err = 1; return; }     /* cannot be a <=252-base read */
        switch (op) {
            case 'M': case '=': case 'X':
                M += num; break;
            case 'I':                                                          /* :321-337 */
                for (uint32_t k = 0; k < num; k++) {
                    if (last_snp) last_snp = md_walk(w, out, M + out.n_ins, read, len);
                    uint32_t at = M + out.n_ins;
                    out.ins(M - prev_i, base_code(at < len ? read[at] : 0u));
                    prev_i = M;
                }
                break;
            case 'D':                                                          /* :340-352 */
                for (uint32_t k = 0; k < num; k++) { out.del(M - prev_d); prev_d = M; }
                break;
            case 'S':
                if (first) {                                                   /* leading clip :358-468 */
                    for (uint32_t k = 0; k < num; k++) {
                        if (last_snp) last_snp = md_walk(w, out, out.n_ins, read, len);
                        out.ins(0u, base_code(k < len ? read[k] : 0u));
                    }
                } else {                                                       /* trailing clip :469-479 */
                    for (uint32_t k = 0; k < num; k++) {
                        uint32_t at = M + out.n_ins;
                        out.ins(M - prev_i, base_code(at < len ? read[at] : 0u));
                        prev_i = M;
                    }
                }
                break;
            case 'H': case 'P': break;
            default: out.err = 1; return;                                      /* '*', 'N', junk */
        }
        if (out.err) return;
        first = 0;
        i = j + 1;
    }
    if (last_snp) md_walk(w, out, len + 1u, read, len);                        /* :551-552 */
    if (out.n_snps > 255u || out.n_dels > 255u || out.n_ins > 255u) out.err = 1;
}

/* 16 bytes from byte offset `off` (any alignment) of a 16-byte-aligned shared array: two aligned 16-byte loads, the
 * word rotation as selects, the byte rotation as funnel shifts (the same fetch as K3's copy path). */
__device__ __forceinline__ uint4 k1_lds16(const uint8_t *base, uint32_t off) {
    const uint4 q0 = *reinterpret_cast<const uint4 *>(base + (off & ~15u));
    const uint4 q1 = *reinterpret_cast<const uint4 *>(base + (off & ~15u) + 16u);
    const bool r2 = (off & 8u) != 0u, r1 = (off & 4u) != 0u;
    const uint32_t x0 = r2 ? q0.z : q0.x, x1 = r2 ? q0.w : q0.y, x2 = r2 ? q1.x : q0.z, x3 = r2 ? q1.y : q0.w,
                   x4 = r2 ? q1.z : q1.x, x5 = r2 ? q1.w : q1.y;
    const uint32_t y0 = r1 ? x1 : x0, y1 = r1 ? x2 : x1, y2 = r1 ? x3 : x2, y3 = r1 ? x4 : x3, y4 = r1 ? x5 : x4;
    const uint32_t sh = (off & 3u) * 8u;
    return make_uint4(__funnelshift_r(y0, y1, sh), __funnelshift_r(y1, y2, sh), __funnelshift_r(y2, y3, sh), __funnelshift_r(y3, y4, sh));
}

struct K1Smem {
    uint64_t bar;
    uint64_t tile_base;
    uint32_t tile;
    uint32_t warp_tot[K1_WARPS];
    uint32_t pos[K1_TILE];
    uint32_t soff[K1_TILE];          /* offset of the read's SEQ in seq[] */
    uint32_t cnt[K1_TILE];           /* n_snps | n_dels << 8 | n_ins << 16 | match << 24 | bad << 25 */
    uint32_t excl[K1_TILE];
    uint32_t roff[K1_TILE];          /* offset of the read's reference bases in ref[] (when in the window) */
    uint16_t len[K1_TILE];
    uint16_t chr_ok[K1_TILE];        /* bit 0: read may use the staged window, bit 1: read passes the input checks */
    uint16_t ecache[K1_TILE][K1_ECACHE];
    __align__(16) uint8_t dyn[16];   /* ref_cap + 64 bytes of reference window, then K1_TILE * max_len + 48 bytes of SEQ (dynamic) */
};

__global__ void __launch_bounds__(K1_TILE)
k1_extract_kernel(DevBatch b, DevGenome g, cbcg_read_rec *__restrict__ recs, uint16_t *__restrict__ edits,
                  uint64_t edits_cap, uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_edits,
                  unsigned long long *err, uint32_t seq_cap, uint32_t ref_cap, uint64_t r_begin, uint64_t r_end, const uint64_t *edit_base) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    K1Smem &S = *reinterpret_cast<K1Smem *>(smem_raw);
    uint8_t *const s_ref = S.dyn, *const s_seq = S.dyn + ref_cap + 64u;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;

    if (tid == 0) {
        S.tile = atomicAdd(ticket, 1u);
        mbar_init(&S.bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    const uint32_t tile = S.tile;
    /* this launch extracts reads [r_begin, r_end): the whole batch, or one chunk of it while the next chunk is still on
       the PCIe link (api.cu); a chunk's edit entries start where the previous chunk's ended (*edit_base). */
    const uint64_t r0 = r_begin + (uint64_t)tile * K1_TILE;
    const uint32_t nr = (uint32_t)min((uint64_t)K1_TILE, r_end - r0);

    /* tile geometry (uniform): SEQ byte range and reference window */
    const uint64_t s0 = b.seq_off[r0], s1 = b.seq_off[r0 + nr];
    const uint64_t a0 = s0 & ~15ull;
    const uint64_t seq_bytes = (s1 - a0 + 15ull) & ~15ull;
    const bool seq_ok = (s1 >= s0) && (seq_bytes <= seq_cap);
    const uint32_t chr0 = b.chr[r0], pos0 = b.pos[r0], chr_l = b.chr[r0 + nr - 1u], pos_l = b.pos[r0 + nr - 1u];
    uint64_t w0 = 0; uint32_t ref_bytes = 0; uint64_t clen0 = 0;
    const uint8_t *ref0 = nullptr;
    if (chr0 < g.n_chr) {
        clen0 = g.chr_len[chr0];
        ref0 = g.bases + g.chr_off[chr0];
        w0 = pos0 ? ((uint64_t)(pos0 - 1u) & ~15ull) : 0ull;
        uint64_t avail = (clen0 + REF_PAD > w0) ? ((clen0 + REF_PAD - w0) & ~15ull) : 0ull;
        ref_bytes = (uint32_t)min((uint64_t)ref_cap, avail);
        /* position-sorted input: the tile's last read bounds the window (a read beyond it takes the HBM path) */
        if (chr_l == chr0 && pos_l >= pos0 && pos0) {
            const uint64_t need = ((uint64_t)(pos_l - 1u) - w0 + b.max_len + 8u + 15u) & ~15ull;
            if (need < ref_bytes) ref_bytes = (uint32_t)need;
        }
    }
    if (tid == 0) {
        uint32_t tx = (seq_ok ? (uint32_t)seq_bytes : 0u) + ref_bytes;
        mbar_expect_tx(&S.bar, tx);
        if (seq_ok && seq_bytes) tma_load_1d(s_seq, b.seq + a0, (uint32_t)seq_bytes, &S.bar);
        if (ref_bytes) tma_load_1d(s_ref, ref0 + w0, ref_bytes, &S.bar);
    }

    /* per-read fixed fields while the copies fly */
    uint32_t my_pos = 0, my_len = 0, my_chr = 0, my_flag = 0;
    uint64_t my_co = 0, my_mo = 0; uint32_t my_clen = 0, my_mlen = 0;
    if (tid < nr) {
        const uint64_t r = r0 + tid;
        my_pos = b.pos[r]; my_len = b.seq_len[r]; my_chr = b.chr[r]; my_flag = b.flag[r];
        const uint64_t so = b.seq_off[r];
        my_co = b.cigar_off[r]; my_clen = (uint32_t)(b.cigar_off[r + 1] - my_co);
        my_mo = b.md_off[r];    my_mlen = (uint32_t)(b.md_off[r + 1] - my_mo);
        S.pos[tid] = my_pos; S.len[tid] = (uint16_t)my_len; S.soff[tid] = (uint32_t)(so - a0);
        bool in_win = (my_chr == chr0) && ref_bytes && my_pos >= 1u && (uint64_t)(my_pos - 1u) >= w0 &&
                      ((uint64_t)(my_pos - 1u) - w0 + my_len + 8u <= ref_bytes);
        bool ok = seq_ok && my_pos >= 1u && my_len >= 1u && my_len <= CBCG_MAX_READ_LEN && my_chr < g.n_chr;
        if (ok) { const uint64_t clen = (my_chr == chr0) ? clen0 : g.chr_len[my_chr]; ok = ((uint64_t)(my_pos - 1u) + my_len <= clen); }
        S.roff[tid] = in_win ? (uint32_t)((uint64_t)(my_pos - 1u) - w0) : 0u;
        S.chr_ok[tid] = (uint16_t)((in_win ? 1u : 0u) | (ok ? 2u : 0u));
    }
    __syncthreads();
    mbar_wait(&S.bar, 0);

    /* ---- phase 1: perfect-match test (src/read_compression.c:291-296). Half a warp per read, 16 bytes per lane:
       SEQ against the staged window, both at arbitrary byte offsets in shared memory. */
    {
        const uint32_t half = lane >> 4, sub = lane & 15u;
        for (uint32_t i0 = warp * 2u; i0 < nr; i0 += K1_WARPS * 2u) {
            const uint32_t i = i0 + half;
            uint32_t diff = 0; bool ok = false;
            if (i < nr) {
                const uint32_t fl = S.chr_ok[i], len = S.len[i], soff = S.soff[i];
                ok = (fl & 2u) != 0u;
                if (ok && (fl & 1u) && len >= 16u) {
                    /* 16-byte pieces at read offsets 0, 16, 32, ... with the last one pulled back to len - 16: every piece
                       lies inside the read, so nothing has to be masked; both sides are fetched at their own alignment */
                    const uint32_t o = min(sub * 16u, len - 16u);
                    if (sub * 16u < len) {
                        const uint4 sv = k1_lds16(s_seq, soff + o), rv = k1_lds16(s_ref, S.roff[i] + o);
                        diff = (sv.x ^ rv.x) | (sv.y ^ rv.y) | (sv.z ^ rv.z) | (sv.w ^ rv.w);
                    }
                } else if (ok) {                          /* window miss: straight from HBM */
                    const uint8_t *rp = g.bases + g.chr_off[b.chr[r0 + i]] + (S.pos[i] - 1u);
                    for (uint32_t j = sub; j < len; j += 16u) diff |= (uint32_t)(s_seq[soff + j] ^ rp[j]);
                }
            }
            const uint32_t bal = __ballot_sync(FULL_MASK, diff != 0u);
            if (sub == 0u && i < nr) S.cnt[i] = (ok && !((bal >> (half * 16u)) & 0xffffu)) ? (1u << 24) : 0u;
        }
    }
    __syncthreads();

    /* ---- phase 2: lane per read, count edits */
    /* (staging the tile's CIGAR / MD text in shared memory as well was measured: 7 % slower, the extra bulk copies and
       the lost CTA per SM cost more than the L1 hits they replace) */
    const uint8_t *my_cig = b.cigar + my_co, *my_md = b.md + my_mo;
    uint32_t my_cnt = 0, my_total = 0;
    if (tid < nr) {
        my_cnt = S.cnt[tid];
        bool bad = !seq_ok || my_pos == 0u || my_len == 0u || my_len > CBCG_MAX_READ_LEN || my_chr >= g.n_chr;
        if (!bad && !(my_cnt >> 24)) {
            EditSink sink = { nullptr, 0u, 0u, 0u, 0u, 0u, 0, S.ecache[tid] };
            walk_read(s_seq + S.soff[tid], my_len, my_cig, my_clen, my_md, my_mlen, sink);
            /* the bases the decoder takes from the reference (len - n_ins aligned, plus the deletions) must lie inside the
               chromosome, as K3 requires: a read whose span runs past the end could not be rebuilt */
            if (!sink.err && (sink.n_ins > my_len ||
                              (uint64_t)(my_pos - 1u) + (my_len - sink.n_ins) + sink.n_dels > g.chr_len[my_chr])) sink.err = 1;
            if (sink.err) bad = true;
            else { my_cnt = sink.n_snps | (sink.n_dels << 8) | (sink.n_ins << 16); my_total = sink.n_snps + sink.n_dels + sink.n_ins; }
        }
        if (bad) { my_cnt = 1u << 25; my_total = 0; dev_set_error(err, CBCG_ERR_INPUT, r0 + tid); }
    }
    /* CTA exclusive scan of my_total */
    uint32_t incl = warp_incl_scan(my_total);
    if (lane == 31) S.warp_tot[warp] = incl;
    __syncthreads();
    uint32_t warp_base = 0, tile_total = 0;
#pragma unroll
    for (uint32_t k = 0; k < K1_WARPS; k++) { uint32_t t = S.warp_tot[k]; if (k < warp) warp_base += t; tile_total += t; }
    const uint32_t my_excl = warp_base + incl - my_total;

    if (warp == 0) {
        uint64_t base = lookback_exclusive(tile_desc, tile, tile_total, err) + (edit_base ? *edit_base : 0ull);
        if (lane == 0) {
            S.tile_base = base;
            if (r0 + nr == r_end) *total_edits = base + tile_total;
        }
    }
    __syncthreads();
    const uint64_t tile_base = S.tile_base;

    /* ---- phase 3: write records and edit entries */
    if (tid < nr) {
        const uint64_t off = tile_base + my_excl;
        __align__(16) cbcg_read_rec rec;
        rec.pos = my_pos; rec.flag = (uint16_t)my_flag; rec.len = (uint16_t)my_len;
        rec.edit_off = (uint32_t)off;
        rec.match = (uint8_t)((my_cnt >> 24) & 1u);
        rec.n_snps = (uint8_t)(my_cnt & 0xffu); rec.n_dels = (uint8_t)((my_cnt >> 8) & 0xffu); rec.n_ins = (uint8_t)((my_cnt >> 16) & 0xffu);
        reinterpret_cast<uint4 *>(recs)[r0 + tid] = *reinterpret_cast<uint4 *>(&rec);
        if (my_total) {
            if (off + my_total > edits_cap) dev_set_error(err, CBCG_ERR_CAPACITY, r0 + tid);
            else if (my_total <= K1_ECACHE) {           /* the count pass kept them: no second walk */
                uint32_t at[3] = { 0u, rec.n_dels, (uint32_t)rec.n_dels + rec.n_snps };
                for (uint32_t k = 0; k < my_total; k++) {
                    const uint32_t e = S.ecache[tid][k], kind = e >> 14;
                    const uint32_t slot = kind == 0u ? at[0]++ : (kind == 1u ? at[1]++ : at[2]++);
                    edits[off + slot] = (uint16_t)(e & 0x3fffu);
                }
            } else {
                EditSink sink = { edits + off, rec.n_dels, rec.n_snps, 0u, 0u, 0u, 0, nullptr };
                walk_read(s_seq + S.soff[tid], my_len, my_cig, my_clen, my_md, my_mlen, sink);
            }
        }
    }
}

void extract_set_carveout(int pct) { cudaFuncSetAttribute(k1_extract_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct); }   /* see k2_coder.cu */

int launch_extract(const DevBatch &b, const DevGenome &g, cbcg_read_rec *recs, uint16_t *edits,
                   uint64_t edits_cap, uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_edits,
                   unsigned long long *err, cudaStream_t st, cudaEvent_t ev_start, cudaEvent_t ev_stop,
                   uint64_t r_begin, uint64_t r_end, const uint64_t *edit_base) {
    if (r_end > b.n_reads) r_end = b.n_reads;
    if (r_begin >= r_end) return 0;
    const uint64_t tiles = extract_num_tiles(r_end - r_begin);
    const uint32_t seq_cap = (K1_TILE * b.max_len + 48u) & ~15u;
    /* reference window: what a tile of position-adjacent reads spans at the batch's coverage, twice over (a read beyond
       the window takes the HBM path); the smaller the window, the more tiles an SM holds */
    const uint32_t ref_cap = b.ref_cap ? std::min<uint32_t>(std::max<uint32_t>((b.ref_cap + 511u) & ~511u, 1024u), K1_REF_CAP) : K1_REF_CAP;
    const size_t smem = sizeof(K1Smem) + ref_cap + 64 + seq_cap + 16;
    /* per device, so no process-wide cache: a context on another GPU of the same process needs it too. The limit is the
       worst case (CBCG_MAX_READ_LEN); occupancy follows the size actually launched with. */
    const size_t smem_max = sizeof(K1Smem) + K1_REF_CAP + 64 + ((K1_TILE * CBCG_MAX_READ_LEN + 48u) & ~15u) + 16;
    if (smem > smem_max) return -1;
    if (cudaFuncSetAttribute(k1_extract_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max) != cudaSuccess) return -1;
    if (cudaMemsetAsync(tile_desc, 0, tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
    if (ev_start) cudaEventRecord(ev_start, st);
    k1_extract_kernel<<<(unsigned)tiles, K1_TILE, smem, st>>>(b, g, recs, edits, edits_cap, tile_desc, ticket,
                                                             total_edits, err, seq_cap, ref_cap, r_begin, r_end, edit_base);
    if (ev_stop) cudaEventRecord(ev_stop, st);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
