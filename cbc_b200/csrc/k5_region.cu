/*
 * k5_region.cu -- K5: region select and compaction (cbcg_decode_region).
 *
 * Runs after the block decoder on the records of a reduced descriptor table (api.cu, "region decode"): a thread per
 * read tests whether the read overlaps one of the query's intervals, and the kept reads' records, chromosome ordinals
 * and container ordinals are written densely, in read order, for K3. The output offsets come from a CTA scan and the
 * same decoupled look-back across tiles as K1 / K3 / K4 (tile order from an atomic ticket).
 *
 *   overlap: pos <= end and pos + span - 1 >= start on the read's chromosome, span = len - n_ins + n_dels (deletions and
 *     insertions are counted per base; the reference codes soft clips as insertions, so clipped bases are not in it).
 *   intervals: sorted by (chromosome, start), overlapping ones merged, so their ends ascend too: the first interval
 *     whose (chromosome, end) is not below (chr, pos) is the only candidate.
 *   ordinals: the reduced table numbers its reads densely; runs[2 k] is the dense ordinal of the first read of run k of
 *     consecutive blocks, runs[2 k + 1] its ordinal in the container.
 */
#include "common.cuh"
#include "internal.h"

#define K5_TILE 256u

uint64_t region_num_tiles(uint64_t n_reads) { return (n_reads + K5_TILE - 1u) / K5_TILE; }

__global__ void __launch_bounds__(K5_TILE)
k5_region_select_kernel(uint64_t n_reads, const cbcg_read_rec *__restrict__ recs, const uint32_t *__restrict__ chr_of,
                        const RegionIv *__restrict__ iv, uint32_t n_iv, const uint64_t *__restrict__ runs, uint32_t n_runs,
                        cbcg_read_rec *__restrict__ out_recs, uint32_t *__restrict__ out_chr, uint64_t *__restrict__ out_ids,
                        uint64_t *tile_desc, uint32_t *ticket, uint64_t *total, unsigned long long *err) {
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp[K5_TILE / 32u];
    __shared__ uint64_t s_base;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t r = (uint64_t)tile * K5_TILE + tid;
    bool keep = false;
    uint4 rec = make_uint4(0u, 0u, 0u, 0u);                       /* cbcg_read_rec as one 16-byte word: pos | flag, len | edit_off | match, n_snps, n_dels, n_ins */
    uint32_t chr = 0;
    if (r < n_reads) {
        rec = reinterpret_cast<const uint4 *>(recs)[r];
        chr = chr_of[r];
        const uint32_t match = rec.w & 0xffu, nd = match ? 0u : (rec.w >> 16) & 0xffu, ni = match ? 0u : rec.w >> 24;
        const uint64_t pos = rec.x, len = rec.y >> 16;
        const uint64_t span = len + nd > ni ? len + nd - ni : 1u;
        const uint64_t last = pos + span - 1u;
        uint32_t lo = 0, hi = n_iv;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            const RegionIv v = iv[mid];
            if (v.chr < chr || (v.chr == chr && v.end < pos)) lo = mid + 1u; else hi = mid;
        }
        keep = pos != 0u && lo < n_iv && iv[lo].chr == chr && iv[lo].start <= last;
    }
    const uint32_t ballot = __ballot_sync(FULL_MASK, keep);
    if (lane == 0) s_warp[warp] = (uint32_t)__popc(ballot);
    __syncthreads();
    uint32_t warp_base = 0, tile_total = 0;
#pragma unroll
    for (uint32_t k = 0; k < K5_TILE / 32u; k++) { const uint32_t t = s_warp[k]; if (k < warp) warp_base += t; tile_total += t; }
    if (warp == 0) {
        const uint64_t base = lookback_exclusive(tile_desc, tile, tile_total, err);
        if (lane == 0) { s_base = base; if ((uint64_t)(tile + 1u) * K5_TILE >= n_reads) *total = base + tile_total; }
    }
    __syncthreads();
    if (!keep) return;
    uint32_t lo = 0, hi = n_runs;                               /* the last run that starts at or below r */
    while (hi - lo > 1u) { const uint32_t mid = (lo + hi) >> 1; if (runs[2u * mid] <= r) lo = mid; else hi = mid; }
    if (!n_runs || runs[2u * lo] > r) { dev_set_error(err, CBCG_ERR_INTERNAL, r); return; }
    const uint64_t at = s_base + warp_base + (uint32_t)__popc(ballot & ((1u << lane) - 1u));
    reinterpret_cast<uint4 *>(out_recs)[at] = rec;
    out_chr[at] = chr;
    out_ids[at] = runs[2u * lo + 1u] + (r - runs[2u * lo]);
}

int launch_region_select(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const RegionIv *iv, uint32_t n_iv,
                         const uint64_t *runs, uint32_t n_runs, cbcg_read_rec *out_recs, uint32_t *out_chr, uint64_t *out_ids,
                         uint64_t *tile_desc, uint32_t *ticket, uint64_t *total, unsigned long long *err, cudaStream_t st) {
    if (cudaMemsetAsync(total, 0, sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (!n_reads) return 0;
    const uint64_t tiles = region_num_tiles(n_reads);
    if (cudaMemsetAsync(tile_desc, 0, tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
    k5_region_select_kernel<<<(unsigned)tiles, K5_TILE, 0, st>>>(n_reads, recs, chr, iv, n_iv, runs, n_runs, out_recs, out_chr,
                                                                 out_ids, tile_desc, ticket, total, err);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
