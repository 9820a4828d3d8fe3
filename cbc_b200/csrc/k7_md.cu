/*
 * k7_md.cu -- K7: the MD of reads that carry none (batches uploaded without MD; cbcg_derive_md).
 *
 * K1 finds a read's mismatches in its MD text. A batch without MD gets one here, while it is made resident: each read's
 * MD is derived from its CIGAR, its SEQ and the reference as uploaded, by md_rule.cuh's rule (the one K6 prints), and
 * written into the batch's MD pool with its md_off entry. K1 and everything after it then run unchanged.
 *
 * A read is checked before its SEQ or its reference is read: the CIGAR parses and uses M I D S H P = X only, its query
 * length (M + I + S + = + X) is the read's length, it deletes at most 255 bases, POS >= 1, the chromosome exists and the
 * reference span (M + = + X + D) ends inside it. A read that fails gets CBCG_ERR_INPUT and an empty MD.
 *
 * B200 design, as K1. One CTA per tile of K7_TILE consecutive reads, a thread per read, tiles in the order of an atomic
 * ticket. The tile's SEQ range and the reference window under its reads are staged into shared memory by two 1-D TMA
 * bulk copies completing on one mbarrier; a read outside the window walks the reference in HBM. A counting pass sizes
 * each read's MD; a CTA scan and a decoupled look-back over tiles (plus *md_base: a chunk's MD continues the previous
 * chunk's) give its offset in the pool; a writing pass emits the text. The last tile writes md_off[r_end] and the exact
 * total of the launch's MD bytes (*total_md).
 *
 * Capacity: a read whose MD does not end inside the pool (md_cap bytes) gets an empty MD at the pool's end (md_off clamped
 * to md_cap) and CBCG_ERR_CAPACITY: no offset ever points past the pool, and *total_md is still exact, so the caller can
 * size the pool and run again.
 */
#include <algorithm>
#include "common.cuh"
#include "internal.h"
#include "md_rule.cuh"

#define K7_TILE    128u
#define K7_WARPS   (K7_TILE / 32u)
#define K7_REF_CAP 8192u          /* most bytes of reference window staged per tile, as K1 */

uint64_t md_num_tiles(uint64_t n_reads) { return (n_reads + K7_TILE - 1) / K7_TILE; }

struct K7Smem {
    uint64_t bar;
    uint64_t tile_base;
    uint32_t tile;
    uint32_t warp_tot[K7_WARPS];
    __align__(16) uint8_t dyn[16];   /* ref_cap + 64 bytes of reference window, then seq_cap bytes of SEQ (dynamic) */
};

/* Reference bases a validated CIGAR aligns to: M + = + X + D. */
__device__ static uint32_t k7_ref_span(const uint8_t *t, uint32_t tl) {
    uint32_t i = 0, span = 0;
    while (i < tl) {
        uint32_t num = 0;
        while (t[i] >= '0' && t[i] <= '9') num = num * 10u + (uint32_t)(t[i++] - '0');
        const uint32_t op = t[i++];
        if (op == 'M' || op == '=' || op == 'X' || op == 'D') span += num;
    }
    return span;
}

__global__ void __launch_bounds__(K7_TILE)
k7_md_kernel(DevBatch b, DevGenome g, uint64_t *__restrict__ md_off, uint8_t *__restrict__ md, uint64_t md_cap,
             uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_md, unsigned long long *err,
             uint32_t seq_cap, uint32_t ref_cap, uint64_t r_begin, uint64_t r_end, const uint64_t *md_base) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    K7Smem &S = *reinterpret_cast<K7Smem *>(smem_raw);
    uint8_t *const s_ref = S.dyn, *const s_seq = S.dyn + ref_cap + 64u;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;

    if (tid == 0) {
        S.tile = atomicAdd(ticket, 1u);
        mbar_init(&S.bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    const uint32_t tile = S.tile;
    const uint64_t r0 = r_begin + (uint64_t)tile * K7_TILE;
    const uint32_t nr = (uint32_t)min((uint64_t)K7_TILE, r_end - r0);

    /* tile geometry (uniform): SEQ byte range and reference window, as K1 */
    const uint64_t s0 = b.seq_off[r0], s1 = b.seq_off[r0 + nr];
    const uint64_t a0 = s0 & ~15ull;
    const uint64_t seq_bytes = (s1 - a0 + 15ull) & ~15ull;
    const bool seq_ok = (s1 >= s0) && (seq_bytes <= seq_cap);
    const uint32_t chr0 = b.chr[r0], pos0 = b.pos[r0], chr_l = b.chr[r0 + nr - 1u], pos_l = b.pos[r0 + nr - 1u];
    uint64_t w0 = 0; uint32_t ref_bytes = 0;
    if (chr0 < g.n_chr) {
        const uint64_t clen0 = g.chr_len[chr0];
        w0 = pos0 ? ((uint64_t)(pos0 - 1u) & ~15ull) : 0ull;
        const uint64_t avail = (clen0 + REF_PAD > w0) ? ((clen0 + REF_PAD - w0) & ~15ull) : 0ull;
        ref_bytes = (uint32_t)min((uint64_t)ref_cap, avail);
        if (chr_l == chr0 && pos_l >= pos0 && pos0) {
            const uint64_t need = ((uint64_t)(pos_l - 1u) - w0 + b.max_len + 8u + 15u) & ~15ull;
            if (need < ref_bytes) ref_bytes = (uint32_t)need;
        }
    }
    if (tid == 0) {
        mbar_expect_tx(&S.bar, (seq_ok ? (uint32_t)seq_bytes : 0u) + ref_bytes);
        if (seq_ok && seq_bytes) tma_load_1d(s_seq, b.seq + a0, (uint32_t)seq_bytes, &S.bar);
        if (ref_bytes) tma_load_1d(s_ref, g.bases + g.chr_off[chr0] + w0, ref_bytes, &S.bar);
    }

    /* the read's checks, while the copies fly: nothing of its SEQ or reference is read before they pass */
    const uint64_t r = r0 + tid;
    const uint8_t *cig = nullptr;
    uint32_t clen = 0, pos = 0, chr = 0, span = 0;
    uint64_t so = 0;
    bool ok = false;
    if (tid < nr) {
        pos = b.pos[r]; chr = b.chr[r]; so = b.seq_off[r];
        const uint64_t co = b.cigar_off[r];
        cig = b.cigar + co; clen = (uint32_t)(b.cigar_off[r + 1] - co);
        ok = pos >= 1u && chr < g.n_chr && k6_cigar_ok(cig, clen, b.seq_len[r]);
        if (ok) { span = k7_ref_span(cig, clen); ok = (uint64_t)(pos - 1u) + span <= g.chr_len[chr]; }
        if (!ok) dev_set_error(err, CBCG_ERR_INPUT, r);
    }
    mbar_wait(&S.bar, 0);
    const bool in_win = ok && chr == chr0 && ref_bytes && (uint64_t)(pos - 1u) >= w0 && (uint64_t)(pos - 1u) - w0 + span <= ref_bytes;
    const uint8_t *seq = seq_ok ? s_seq + (so - a0) : b.seq + so;
    const uint8_t *ref = in_win ? s_ref + ((uint64_t)(pos - 1u) - w0) : (ok ? g.bases + g.chr_off[chr] + (pos - 1u) : nullptr);

    /* counting pass */
    uint32_t len = 0, nm = 0;
    if (ok) { K6Out<false> o{ nullptr, 0u }; k6_md_walk(o, cig, clen, seq, ref, &nm); len = o.n; }

    /* offsets: CTA scan, look-back across tiles */
    const uint32_t incl = warp_incl_scan(len);
    if (lane == 31u) S.warp_tot[warp] = incl;
    __syncthreads();
    uint32_t warp_base = 0, tile_total = 0;
#pragma unroll
    for (uint32_t k = 0; k < K7_WARPS; k++) { const uint32_t t = S.warp_tot[k]; if (k < warp) warp_base += t; tile_total += t; }
    if (warp == 0) {
        const uint64_t base = lookback_exclusive(tile_desc, tile, tile_total, err) + (md_base ? *md_base : 0ull);
        if (lane == 0) {
            S.tile_base = base;
            if (r0 + nr == r_end) *total_md = base + tile_total;
        }
    }
    __syncthreads();

    /* writing pass */
    if (tid < nr) {
        const uint64_t off = S.tile_base + warp_base + incl - len;
        const bool fits = off + len <= md_cap;
        md_off[r] = fits ? off : md_cap;
        if (r + 1u == r_end) md_off[r_end] = min(off + len, md_cap);
        if (!fits) dev_set_error(err, CBCG_ERR_CAPACITY, r);
        else if (len) { K6Out<true> o{ md + off, 0u }; k6_md_walk(o, cig, clen, seq, ref, &nm); }
    }
}

int launch_md(const DevBatch &b, const DevGenome &g, uint64_t *md_off, uint8_t *md, uint64_t md_cap, uint64_t *tile_desc,
              uint32_t *ticket, uint64_t *total_md, unsigned long long *err, cudaStream_t st, uint64_t r_begin, uint64_t r_end,
              const uint64_t *md_base) {
    if (r_end > b.n_reads) r_end = b.n_reads;
    if (r_begin >= r_end) return 0;
    if (b.max_len == 0 || b.max_len > CBCG_MAX_READ_LEN) return -1;
    const uint64_t tiles = md_num_tiles(r_end - r_begin);
    const uint32_t seq_cap = (K7_TILE * b.max_len + 48u) & ~15u;
    const uint32_t ref_cap = b.ref_cap ? std::min<uint32_t>(std::max<uint32_t>((b.ref_cap + 511u) & ~511u, 1024u), K7_REF_CAP) : K7_REF_CAP;
    const size_t smem = sizeof(K7Smem) + ref_cap + 64 + seq_cap;
    const size_t smem_max = sizeof(K7Smem) + K7_REF_CAP + 64 + ((K7_TILE * CBCG_MAX_READ_LEN + 48u) & ~15u);
    if (cudaFuncSetAttribute(k7_md_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max) != cudaSuccess) return -1;
    if (cudaMemsetAsync(tile_desc, 0, tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
    k7_md_kernel<<<(unsigned)tiles, K7_TILE, smem, st>>>(b, g, md_off, md, md_cap, tile_desc, ticket, total_md, err, seq_cap, ref_cap,
                                                        r_begin, r_end, md_base);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
