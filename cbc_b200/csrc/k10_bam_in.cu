/*
 * k10_bam_in.cu -- K10: BAM input (cbcg_bgzf_inflate, cbcg_bam_open, cbcg_batch_upload_bam; DESIGN.md 5g).
 *
 * BGZF members (SAMv1 4.1) are independent raw deflate streams (RFC 1951) of at most 64 KiB of output each. The host walks
 * the chain of member headers (no payload read) and gives every member its output offset, an exclusive scan of ISIZE. Then:
 *
 *   k10_inflate_kernel: one warp per member. Lane 0 decodes the bit stream: stored, fixed and dynamic Huffman blocks, any
 *     number of them; each code is a canonical code held in shared memory as a count per length, its symbols in code order
 *     and a primary table of K10_PBITS bits, so codes up to K10_PBITS bits resolve with one look-up and longer ones (to 15
 *     bits) by the canonical walk over the counts. Lane 0 writes literals itself and queues matches and stored blocks; when
 *     the queue is full or the member ends, the warp copies the queue in order, 32 bytes per step (byte j of
 *     a match <len, dist> at out p is out[p - dist + j mod dist], so overlapping matches need no serial copy). Every read of
 *     compressed input and every write of output is checked against the member's extent; a bad block type, a code that is
 *     over-subscribed or incomplete, a distance before the member's start, a length or distance symbol outside the alphabet,
 *     running out of input or writing past ISIZE is CBCG_ERR_CORRUPT for the member, never an access outside it. The warp
 *     then checks ISIZE and computes the CRC32 of the member's output (a chunk per lane, combined by GF(2) shifts, bgzf.cuh).
 *
 *   record boundaries, exact and parallel. The inflated stream (the caller's carry, then the members) is cut into segments,
 *     one per member (segment 0 also holds the carry). k10_guess_kernel: a warp per segment finds the first offset that
 *     passes k10_plausible -- a test every real record passes -- 32 offsets per step (segment 0 starts at offset 0, a known
 *     record start), and lane 0 walks the block_size chain from it to the first record that starts past the segment,
 *     counting the whole records. A walk stops at a block_size below 32 (no record has one), so every record it passes is
 *     at least 36 bytes: a stream of T bytes holds at most T / 36 of them, which sizes the record-offset array; a true
 *     chain that meets such a block_size is CBCG_ERR_FORMAT. k10_chain_kernel (one warp) then proves the chain: the true entry of segment k is the true
 *     exit of segment k - 1; where the guess equals it, the walk stands; where it does not (a decoy, or a record cut by the
 *     end of the input), the segment is walked again from the true entry. A segment in which no record starts passes the
 *     entry through. The warp loads 32 segments' results at once and resolves them in order with shuffles, so the serial
 *     part costs a few instructions per member, not a load per record. k10_rec_start_kernel writes every whole record's
 *     offset, a thread per segment.
 *
 *   k10_count_kernel: a thread per record, tiles of K10_TILE from an atomic ticket. Checks the record's layout, skips FLAG & 4
 *     (counted as unmapped), maps refID through the host's map to the loaded-reference ordinal, sizes SEQ, the CIGAR text
 *     ("%u%c" per operation, "*" for none) and the MD:Z payload (a walk over the aux fields of every type); a CTA scan and
 *     four decoupled look-backs give each mapped record its read ordinal and its offsets in the three pools, written straight
 *     into the resident batch's arrays with POS, FLAG, the length and the chromosome. k10_write_kernel: a thread per read
 *     writes SEQ (the 4-bit code spelled =ACMGRSVTWYHKDBN), the CIGAR text and MD, and lists where the chromosome changes.
 */
#include "common.cuh"
#include "internal.h"
#include "bgzf.cuh"

#define K10_WARPS 4u                      /* members per CTA */
#define K10_Q 64u                         /* queued matches / stored blocks per warp */
#define K10_PBITS 9u                      /* primary table bits */
#define K10_TILE 128u
#define K10_NONE (~0ull)

/* ---------------------------------------------------------------- inflate */
static __constant__ uint16_t k10_lbase[29] = { 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115,
                                               131, 163, 195, 227, 258 };
static __constant__ uint8_t k10_lext[29] = { 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0 };
static __constant__ uint16_t k10_dbase[30] = { 1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537,
                                               2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577 };
static __constant__ uint8_t k10_dext[30] = { 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13 };
static __constant__ uint8_t k10_clorder[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

struct K10Huff {
    uint16_t count[16];                   /* codes per length */
    uint16_t sym[288];                    /* symbols by (length, symbol) */
    uint16_t prim[1u << K10_PBITS];       /* symbol << 4 | length for codes of <= K10_PBITS bits; 0: longer (or unused) */
};
struct K10Tok { uint32_t out, len, src; };     /* src: distance, or K10_STORED | input offset in the member */
#define K10_STORED 0x80000000u
struct K10Warp {
    K10Huff lit, dist;
    uint16_t lens[320];
    K10Tok q[K10_Q];
    uint32_t qn, done;
};

/* LSB-first bit reader over the member's deflate bytes [0, end). Past the end it feeds zeros; overrun() tells when a
   consumed bit was one of them. */
struct K10Bits {
    const uint8_t *p; uint32_t pos, end; uint64_t buf; uint32_t cnt;
    __device__ __forceinline__ void refill() {
        while (cnt <= 56u) { const uint64_t b = pos < end ? (uint64_t)__ldg(p + pos) : 0ull; pos++; buf |= b << cnt; cnt += 8u; }
    }
    __device__ __forceinline__ uint32_t bits(uint32_t n) {   /* n <= 32 */
        refill();
        const uint32_t v = (uint32_t)(buf & ((1ull << n) - 1ull));
        buf >>= n; cnt -= n;
        return v;
    }
    __device__ __forceinline__ bool overrun() const { return (uint64_t)pos * 8u - cnt > (uint64_t)end * 8u; }
};

/* The canonical code of lengths len[0, n): 0 ok, -1 over-subscribed, or incomplete where that is not allowed (an
   incomplete code is allowed only when it is a single code of one bit, as zlib's inflate_table; the code-length code
   never). A code without symbols is built empty: decoding from it fails. */
__device__ static int k10_build(K10Huff &h, const uint16_t *len, uint32_t n, bool codes) {
    for (uint32_t l = 0; l < 16u; l++) h.count[l] = 0;
    for (uint32_t s = 0; s < n; s++) h.count[len[s]]++;
    for (uint32_t k = 0; k < (1u << K10_PBITS); k++) h.prim[k] = 0;
    if (h.count[0] == n) return 0;
    int left = 1; uint32_t max = 0;
    for (uint32_t l = 1; l < 16u; l++) { left <<= 1; left -= h.count[l]; if (left < 0) return -1; if (h.count[l]) max = l; }
    if (left > 0 && (codes || max != 1u)) return -1;
    uint16_t offs[16];
    offs[1] = 0;
    for (uint32_t l = 1; l < 15u; l++) offs[l + 1] = offs[l] + h.count[l];
    for (uint32_t s = 0; s < n; s++) if (len[s]) h.sym[offs[len[s]]++] = (uint16_t)s;
    uint32_t code = 0, i = 0;
    for (uint32_t l = 1; l <= K10_PBITS; l++) {
        for (uint32_t c = 0; c < h.count[l]; c++, i++, code++) {
            const uint32_t rev = __brev(code) >> (32u - l);
            for (uint32_t k = rev; k < (1u << K10_PBITS); k += 1u << l) h.prim[k] = (uint16_t)(h.sym[i] << 4 | l);
        }
        code <<= 1;
    }
    return 0;
}
/* one symbol, or -1 */
__device__ __forceinline__ int k10_decode(K10Bits &b, const K10Huff &h) {
    b.refill();
    const uint32_t e = h.prim[b.buf & ((1u << K10_PBITS) - 1u)];
    if (e) { const uint32_t l = e & 15u; b.buf >>= l; b.cnt -= l; return (int)(e >> 4); }
    uint64_t bits = b.buf;
    int code = 0, first = 0, index = 0;
    for (uint32_t len = 1; len < 16u; len++) {
        code |= (int)(bits & 1u); bits >>= 1;
        const int count = h.count[len];
        if (code - count < first) { b.buf >>= len; b.cnt -= len; return h.sym[index + (code - first)]; }
        index += count; first += count; first <<= 1; code <<= 1;
    }
    return -1;
}

/* Lane 0's decoder state between queue flushes. */
struct K10State { uint32_t opos; uint32_t in_block; uint32_t last; uint32_t bad; };

/* Decode until the queue is full, the block ends or the member ends (lane 0). out: the member's output, isize bytes. */
__device__ static void k10_step(K10Warp &W, K10Bits &b, K10State &s, uint8_t *out, uint32_t isize) {
    uint32_t qn = 0;
    while (!s.bad && qn < K10_Q) {
        if (!s.in_block) {
            if (s.last) { W.done = 1; break; }
            s.last = b.bits(1);
            const uint32_t type = b.bits(2);
            if (type == 0u) {                              /* stored: to the byte, LEN, NLEN, the bytes */
                const uint32_t drop = b.cnt & 7u; b.buf >>= drop; b.cnt -= drop;
                const uint32_t len = b.bits(16), nlen = b.bits(16);
                if (b.overrun() || (len ^ 0xffffu) != nlen) { s.bad = 1; break; }
                const uint32_t at = b.pos - b.cnt / 8u;    /* the whole bytes still in the buffer were not consumed */
                if (at + len > b.end || s.opos + len > isize) { s.bad = 1; break; }
                if (len) { W.q[qn++] = K10Tok{ s.opos, len, K10_STORED | at }; s.opos += len; }
                b.pos = at + len; b.buf = 0; b.cnt = 0;
                continue;
            }
            if (type == 3u) { s.bad = 1; break; }
            if (type == 1u) {                              /* fixed Huffman */
                for (uint32_t k = 0; k < 288u; k++) W.lens[k] = k < 144u ? 8u : k < 256u ? 9u : k < 280u ? 7u : 8u;
                k10_build(W.lit, W.lens, 288u, false);
                for (uint32_t k = 0; k < 32u; k++) W.lens[k] = 5u;
                k10_build(W.dist, W.lens, 32u, false);
            } else {                                       /* dynamic Huffman */
                const uint32_t hlit = b.bits(5) + 257u, hdist = b.bits(5) + 1u, hclen = b.bits(4) + 4u;
                if (hlit > 286u || hdist > 30u) { s.bad = 1; break; }
                for (uint32_t k = 0; k < 19u; k++) W.lens[k] = 0;
                for (uint32_t k = 0; k < hclen; k++) W.lens[k10_clorder[k]] = (uint16_t)b.bits(3);
                if (k10_build(W.lit, W.lens, 19u, true)) { s.bad = 1; break; }
                uint32_t n = 0;
                while (n < hlit + hdist) {
                    const int sym = k10_decode(b, W.lit);
                    if (sym < 0) { s.bad = 1; break; }
                    if (sym < 16) { W.lens[n++] = (uint16_t)sym; continue; }
                    uint32_t l = 0, rep;
                    if (sym == 16) { if (n == 0) { s.bad = 1; break; } l = W.lens[n - 1]; rep = 3u + b.bits(2); }
                    else if (sym == 17) rep = 3u + b.bits(3);
                    else rep = 11u + b.bits(7);
                    if (n + rep > hlit + hdist) { s.bad = 1; break; }
                    while (rep--) W.lens[n++] = (uint16_t)l;
                }
                if (s.bad || b.overrun() || W.lens[256] == 0) { s.bad = 1; break; }
                if (k10_build(W.lit, W.lens, hlit, false) || k10_build(W.dist, W.lens + hlit, hdist, false)) { s.bad = 1; break; }
            }
            s.in_block = 1;
        }
        /* symbols of a Huffman block */
        for (;;) {
            const int sym = k10_decode(b, W.lit);
            if (sym < 0) { s.bad = 1; break; }
            if (sym < 256) {
                if (s.opos >= isize) { s.bad = 1; break; }
                out[s.opos++] = (uint8_t)sym;
                continue;
            }
            if (sym == 256) { s.in_block = 0; break; }
            const uint32_t li = (uint32_t)sym - 257u;
            if (li >= 29u) { s.bad = 1; break; }
            const uint32_t len = k10_lbase[li] + b.bits(k10_lext[li]);
            const int ds = k10_decode(b, W.dist);
            if (ds < 0 || ds >= 30) { s.bad = 1; break; }
            const uint32_t dist = k10_dbase[ds] + b.bits(k10_dext[ds]);
            if (dist > s.opos || s.opos + len > isize) { s.bad = 1; break; }
            W.q[qn++] = K10Tok{ s.opos, len, dist };
            s.opos += len;
            if (qn == K10_Q) break;
        }
        if (b.overrun()) s.bad = 1;
    }
    if (s.bad) W.done = 1;
    W.qn = qn;
}

__global__ void __launch_bounds__(32u * K10_WARPS)
k10_inflate_kernel(const uint8_t *__restrict__ in, const BgzfMember *__restrict__ mem, uint32_t n_members, uint8_t *__restrict__ out,
                   unsigned long long *err) {
    __shared__ K10Warp sw[K10_WARPS];
    __shared__ uint32_t crc_tab[256];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t k = threadIdx.x; k < 256u; k += blockDim.x) crc_tab[k] = bgzf_crc_table_entry(k);
    __syncthreads();
    const uint32_t m = blockIdx.x * K10_WARPS + warp;
    if (m >= n_members) return;
    K10Warp &W = sw[warp];
    const BgzfMember M = mem[m];
    uint8_t *o = out + M.out_off;
    const uint8_t *src = in + M.in_off;
    K10Bits b{ src, 0u, M.in_len, 0ull, 0u };
    K10State s{ 0u, 0u, 0u, 0u };
    if (lane == 0) W.done = 0;
    __syncwarp();
    for (;;) {
        if (lane == 0) k10_step(W, b, s, o, M.isize);
        __syncwarp();
        const uint32_t qn = W.qn;
        for (uint32_t t = 0; t < qn; t++) {
            const K10Tok k = W.q[t];
            if (k.src & K10_STORED) {
                const uint8_t *from = src + (k.src & ~K10_STORED);
                for (uint32_t j = lane; j < k.len; j += 32u) o[k.out + j] = from[j];
            } else {
                for (uint32_t j = lane; j < k.len; j += 32u) o[k.out + j] = o[k.out - k.src + j % k.src];
            }
            __syncwarp();
        }
        const uint32_t done = W.done;
        __syncwarp();
        if (done) break;
    }
    const uint32_t bad = __shfl_sync(FULL_MASK, s.bad | (s.opos != M.isize ? 1u : 0u), 0);
    if (bad) { if (lane == 0) dev_set_error(err, CBCG_ERR_CORRUPT, m); return; }
    const uint32_t B = M.isize, ch = (B + 31u) / 32u;
    const uint32_t a = min(B, lane * ch), e = min(B, a + ch);
    uint32_t crc = 0;
    for (uint32_t p = a; p < e; p++) crc = crc_tab[(crc ^ o[p]) & 0xffu] ^ (crc >> 8);
    uint32_t part = a < e ? bgzf_crc_shift(crc, B - e) : 0u;
    for (int x = 16; x > 0; x >>= 1) part ^= __shfl_xor_sync(FULL_MASK, part, x);
    if (lane == 0 && bgzf_crc_finish(part, B) != M.crc) dev_set_error(err, CBCG_ERR_CORRUPT, m);
}

int launch_inflate(const uint8_t *in, const BgzfMember *mem, uint32_t n_members, uint8_t *out, unsigned long long *err, cudaStream_t st) {
    if (!n_members) return 0;
    k10_inflate_kernel<<<(n_members + K10_WARPS - 1u) / K10_WARPS, 32u * K10_WARPS, 0, st>>>(in, mem, n_members, out, err);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

/* ---------------------------------------------------------------- record boundaries */
__device__ __forceinline__ uint32_t k10_u32(const uint8_t *s, uint64_t p) {
    return (uint32_t)s[p] | (uint32_t)s[p + 1] << 8 | (uint32_t)s[p + 2] << 16 | (uint32_t)s[p + 3] << 24;
}
__device__ __forceinline__ uint32_t k10_u16(const uint8_t *s, uint64_t p) { return (uint32_t)s[p] | (uint32_t)s[p + 1] << 8; }

/* A test every BAM record (SAMv1 4.2) passes: block_size >= 32, refID and next refID in [-1, n_ref), l_read_name >= 1 with
   the name's characters in '!'..'~' and a NUL at its end, and the fixed fields, name, CIGAR, SEQ and QUAL inside block_size. */
__device__ static bool k10_plausible(const uint8_t *s, uint64_t p, uint64_t T, int32_t n_ref) {
    if (p + 36u > T) return false;
    const uint32_t bs = k10_u32(s, p);
    if (bs < 32u) return false;
    const int32_t ref = (int32_t)k10_u32(s, p + 4), nref = (int32_t)k10_u32(s, p + 24), l_seq = (int32_t)k10_u32(s, p + 20);
    if (ref < -1 || ref >= n_ref || nref < -1 || nref >= n_ref || l_seq < 0) return false;
    const uint32_t lrn = s[p + 12], n_cig = k10_u16(s, p + 16);
    if (lrn < 1u) return false;
    if (32ull + lrn + 4ull * n_cig + ((uint64_t)l_seq + 1u) / 2u + (uint64_t)l_seq > bs) return false;
    if (p + 36u + lrn > T) return false;
    for (uint32_t i = 0; i + 1u < lrn; i++) { const uint8_t c = s[p + 36u + i]; if (c < '!' || c > '~') return false; }
    return s[p + 35u + lrn] == 0u;
}
/* The record after the one at p, or K10_NONE when the one at p does not end inside the stream (the tail) or is malformed:
   block_size < 32, which no record has. Every record a chain passes is therefore at least 36 bytes long. */
__device__ __forceinline__ uint64_t k10_next(const uint8_t *s, uint64_t p, uint64_t T) {
    if (p + 4u > T) return K10_NONE;
    const uint32_t bs = k10_u32(s, p);
    const uint64_t nx = p + 4u + bs;
    return (bs < 32u || nx > T) ? K10_NONE : nx;
}
/* 1 when the chain stopped at p because of a malformed record there, not because the stream ends inside it */
__device__ __forceinline__ bool k10_malformed(const uint8_t *s, uint64_t p, uint64_t T) { return p + 4u <= T && k10_u32(s, p) < 32u; }
/* The block_size chain from a record start p to the first record that starts at or past hi, or to the first record that
   does not end inside the stream or is malformed. Returns where it stopped; *n: the whole records passed. */
__device__ static uint64_t k10_walk(const uint8_t *s, uint64_t p, uint64_t hi, uint64_t T, uint64_t *n) {
    uint64_t c = 0;
    while (p < hi) {
        const uint64_t nx = k10_next(s, p, T);
        if (nx == K10_NONE) break;
        c++; p = nx;
    }
    *n = c;
    return p;
}

/* a warp per segment: its guess, and the walk from it (exit, whole records) */
__global__ void __launch_bounds__(128)
k10_guess_kernel(const uint8_t *__restrict__ s, uint64_t T, const uint64_t *__restrict__ seg, uint32_t n_seg, int32_t n_ref,
                 uint64_t *guess, uint64_t *exit_, uint64_t *count) {
    const uint32_t lane = threadIdx.x & 31u, k = blockIdx.x * 4u + (threadIdx.x >> 5);
    if (k >= n_seg) return;
    const uint64_t lo = seg[k], hi = seg[k + 1];
    uint64_t g = K10_NONE;
    if (k == 0) g = lo < hi ? 0ull : K10_NONE;
    else
        for (uint64_t b = lo; b < hi; b += 32u) {
            const bool ok = b + lane < hi && k10_plausible(s, b + lane, T, n_ref);
            const uint32_t v = __ballot_sync(FULL_MASK, ok);
            if (v) { g = b + (uint32_t)(__ffs(v) - 1); break; }
        }
    if (lane) return;
    uint64_t n = 0, x = K10_NONE;
    if (g != K10_NONE) x = k10_walk(s, g, hi, T, &n);
    guess[k] = g; exit_[k] = x; count[k] = n;
}

/* One warp proves the chain segment by segment: entry[k] (K10_NONE: no whole record starts in it) and base[k], the
   ordinal of its first record. words: [0] whole records, [1] the tail's start, [2] segments walked again. A chain that
   meets a record with block_size < 32 stops there: CBCG_ERR_FORMAT, item the record's ordinal. */
__global__ void __launch_bounds__(32)
k10_chain_kernel(const uint8_t *__restrict__ s, uint64_t T, const uint64_t *__restrict__ seg, uint32_t n_seg, const uint64_t *guess,
                 const uint64_t *exit_, const uint64_t *count, uint64_t *entry, uint64_t *base, uint64_t *words, unsigned long long *err) {
    const uint32_t lane = threadIdx.x;
    uint64_t X = 0, nrec = 0, repairs = 0;
    bool ended = false;                                   /* the chain reached a record that does not end in the stream */
    for (uint32_t k0 = 0; k0 < n_seg; k0 += 32u) {
        const uint32_t k = k0 + lane;
        uint64_t g = K10_NONE, x = K10_NONE, c = 0, hi = T;
        if (k < n_seg) { g = guess[k]; x = exit_[k]; c = count[k]; hi = seg[k + 1]; }
        uint64_t my_entry = K10_NONE, my_base = 0;
        const uint32_t n = min(32u, n_seg - k0);
        for (uint32_t j = 0; j < n; j++) {
            const uint64_t gj = __shfl_sync(FULL_MASK, g, j), xj = __shfl_sync(FULL_MASK, x, j), cj = __shfl_sync(FULL_MASK, c, j);
            const uint64_t hj = __shfl_sync(FULL_MASK, hi, j);
            uint64_t E = K10_NONE, cnt = 0;
            if (!ended && X < hj) {                        /* a record starts in segment j: X */
                E = X;
                if (gj == X) { cnt = cj; X = xj; }
                else { X = k10_walk(s, X, hj, T, &cnt); repairs++; }
                if (X < hj) {                              /* stopped inside the segment: the tail starts at X, or a malformed record */
                    ended = true;
                    if (lane == 0 && k10_malformed(s, X, T)) dev_set_error(err, CBCG_ERR_FORMAT, nrec + cnt);
                }
            }
            if (lane == j) { my_entry = E; my_base = nrec; }
            nrec += cnt;
        }
        if (k < n_seg) { entry[k] = my_entry; base[k] = my_base; }
    }
    if (lane == 0) { words[0] = nrec; words[1] = X < T ? X : T; words[2] = repairs; }
}

/* a thread per segment: the offset of every whole record, by ordinal (rec_cap entries; the chain's records are >= 36
   bytes each, so T / 36 + 1 always suffice -- the check keeps any disagreement from writing past the array) */
__global__ void k10_rec_start_kernel(const uint8_t *__restrict__ s, uint64_t T, const uint64_t *__restrict__ seg, uint32_t n_seg,
                                     const uint64_t *__restrict__ entry, const uint64_t *__restrict__ base, uint64_t *rec_start,
                                     uint64_t rec_cap, unsigned long long *err) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_seg || entry[k] == K10_NONE) return;
    uint64_t p = entry[k], i = base[k];
    const uint64_t hi = seg[k + 1];
    while (p < hi) {
        const uint64_t nx = k10_next(s, p, T);
        if (nx == K10_NONE) break;
        if (i >= rec_cap) { dev_set_error(err, CBCG_ERR_INTERNAL, i); return; }
        rec_start[i++] = p; p = nx;
    }
}

int launch_bam_boundaries(const uint8_t *stream, uint64_t T, const uint64_t *seg, uint32_t n_seg, int32_t n_ref, uint64_t *work,
                          uint64_t *rec_start, uint64_t rec_cap, uint64_t *words, unsigned long long *err, cudaStream_t st) {
    if (!n_seg) return 0;
    uint64_t *guess = work, *exit_ = work + n_seg, *count = work + 2ull * n_seg, *entry = work + 3ull * n_seg, *base = work + 4ull * n_seg;
    k10_guess_kernel<<<(n_seg + 3u) / 4u, 128, 0, st>>>(stream, T, seg, n_seg, n_ref, guess, exit_, count);
    k10_chain_kernel<<<1, 32, 0, st>>>(stream, T, seg, n_seg, guess, exit_, count, entry, base, words, err);
    k10_rec_start_kernel<<<(n_seg + 127u) / 128u, 128, 0, st>>>(stream, T, seg, n_seg, entry, base, rec_start, rec_cap, err);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

/* ---------------------------------------------------------------- record parse */
__device__ __forceinline__ uint32_t k10_digits(uint32_t v) {
    uint32_t d = 1;
    while (v >= 10u) { v /= 10u; d++; }
    return d;
}
/* aux field value sizes; 0: Z / H (to the NUL), B (array), or not a type */
__device__ __forceinline__ uint32_t k10_aux_size(uint32_t t) {
    return (t == 'A' || t == 'c' || t == 'C') ? 1u : (t == 's' || t == 'S') ? 2u : (t == 'i' || t == 'I' || t == 'f') ? 4u : 0u;
}

/* The MD:Z payload among the aux fields [a, e): its offset and length, 0 when absent, -1 when the fields are malformed. */
__device__ static int k10_find_md(const uint8_t *s, uint64_t a, uint64_t e, uint64_t *md, uint32_t *md_len) {
    while (a < e) {
        if (a + 3u > e) return -1;
        const uint8_t t0 = s[a], t1 = s[a + 1], ty = s[a + 2];
        a += 3u;
        const uint32_t fixed = k10_aux_size(ty);
        if (fixed) { a += fixed; continue; }
        if (ty == 'Z' || ty == 'H') {
            const uint64_t v = a;
            while (a < e && s[a]) a++;
            if (a >= e) return -1;
            if (t0 == 'M' && t1 == 'D' && ty == 'Z') { *md = v; *md_len = (uint32_t)(a - v); return 1; }
            a++;
            continue;
        }
        if (ty == 'B') {
            if (a + 5u > e) return -1;
            const uint32_t sz = k10_aux_size(s[a]);
            if (!sz || s[a] == 'A') return -1;
            a += 5u + (uint64_t)sz * k10_u32(s, a + 1);
            continue;
        }
        return -1;
    }
    return a == e ? 0 : -1;
}

struct K10Rec { uint64_t p; uint32_t mapped, seq, cig, md, chr, pos, flag; uint64_t md_at; };

/* the record at p (ordinal r): checks, sizes; errors are set here */
__device__ static K10Rec k10_read(const uint8_t *s, uint64_t p, uint64_t r, const int32_t *map, int32_t n_ref, uint32_t derive,
                                  unsigned long long *err, uint32_t *len_slot) {
    K10Rec R{};
    R.p = p;
    const uint32_t bs = k10_u32(s, p);
    const int32_t ref = (int32_t)k10_u32(s, p + 4), l_seq = (int32_t)k10_u32(s, p + 20);
    const uint32_t lrn = s[p + 12], n_cig = k10_u16(s, p + 16), flag = k10_u16(s, p + 18);
    const uint64_t fixed = 32ull + lrn + 4ull * n_cig + ((uint64_t)(uint32_t)l_seq + 1u) / 2u + (uint64_t)(uint32_t)l_seq;
    if (bs < 32u || lrn < 1u || l_seq < 0 || fixed > bs) { dev_set_error(err, CBCG_ERR_FORMAT, r); return R; }
    if (r < 2u) len_slot[r] = (uint32_t)l_seq;
    if (flag & 4u) return R;                               /* unmapped: counted, not kept (src/compression.c:50) */
    const int32_t chr = (ref >= 0 && ref < n_ref) ? map[ref] : -1;
    if (chr < 0) { dev_set_error(err, CBCG_ERR_NO_REFERENCE, r); return R; }
    if (l_seq == 0 || l_seq > 0xffff) { dev_set_error(err, CBCG_ERR_INPUT, r); return R; }
    const uint64_t c0 = p + 36u + lrn;
    uint32_t cig = n_cig ? 0u : 1u;                        /* "*" */
    for (uint32_t k = 0; k < n_cig; k++) {
        const uint32_t v = k10_u32(s, c0 + 4ull * k);
        if ((v & 15u) > 8u) { dev_set_error(err, CBCG_ERR_FORMAT, r); return R; }
        cig += k10_digits(v >> 4) + 1u;
    }
    if (!derive) {
        uint64_t md = 0; uint32_t ml = 0;
        const int f = k10_find_md(s, c0 + 4ull * n_cig + ((uint32_t)l_seq + 1u) / 2u + (uint32_t)l_seq, p + 4u + bs, &md, &ml);
        if (f < 0) { dev_set_error(err, CBCG_ERR_FORMAT, r); return R; }
        if (f == 0) { dev_set_error(err, CBCG_ERR_INPUT, r); return R; }
        R.md = ml; R.md_at = md;
    }
    R.mapped = 1; R.seq = (uint32_t)l_seq; R.cig = cig; R.chr = (uint32_t)chr;
    R.pos = k10_u32(s, p + 8) + 1u; R.flag = flag;
    return R;
}

struct K10Smem { uint32_t tile; uint32_t wt[4][K10_TILE / 32u]; uint64_t base[4]; };

/* sizes, ordinals and offsets of the mapped records; POS, FLAG, length and chromosome into the batch; src[o] / md_at[o]:
   the record and its MD payload. words: [3] reads, [4] SEQ, [5] CIGAR, [6] MD bytes; lens: [0] [1] l_seq of records 0 and
   1, [2] 0xffffffff - shortest, [3] longest read. */
__global__ void __launch_bounds__(K10_TILE)
k10_count_kernel(const uint8_t *__restrict__ s, const uint64_t *__restrict__ rec_start, uint64_t n_rec, const int32_t *__restrict__ map,
                 int32_t n_ref, uint32_t derive, uint32_t *pos, uint16_t *flag, uint16_t *seq_len, uint32_t *chr, uint64_t *seq_off,
                 uint64_t *cigar_off, uint64_t *md_off, uint64_t *src, uint64_t *md_at, uint64_t *desc, uint32_t *ticket, uint64_t *words,
                 uint32_t *lens, unsigned long long *err) {
    __shared__ K10Smem S;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) S.tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = S.tile;
    const uint64_t n_tiles = (n_rec + K10_TILE - 1u) / K10_TILE;
    const uint64_t r = (uint64_t)tile * K10_TILE + tid;
    K10Rec R{};
    if (r < n_rec) R = k10_read(s, rec_start[r], r, map, n_ref, derive, err, lens);
    const uint32_t v[4] = { R.mapped, R.seq, R.cig, R.md };
    uint32_t incl[4];
#pragma unroll
    for (int q = 0; q < 4; q++) { incl[q] = warp_incl_scan(v[q]); if (lane == 31u) S.wt[q][warp] = incl[q]; }
    if (R.mapped) { atomicMax(&lens[2], 0xffffffffu - R.seq); atomicMax(&lens[3], R.seq); }
    __syncthreads();
    uint32_t wb[4] = { 0, 0, 0, 0 }, tot[4] = { 0, 0, 0, 0 };
#pragma unroll
    for (int q = 0; q < 4; q++)
        for (uint32_t k = 0; k < K10_TILE / 32u; k++) { const uint32_t t = S.wt[q][k]; if (k < warp) wb[q] += t; tot[q] += t; }
    if (warp == 0) {
#pragma unroll
        for (int q = 0; q < 4; q++) { const uint64_t b = lookback_exclusive(desc + q * n_tiles, tile, tot[q], err); if (lane == 0) S.base[q] = b; }
    }
    __syncthreads();
    if (r < n_rec && R.mapped) {
        const uint64_t o = S.base[0] + wb[0] + incl[0] - 1u;
        pos[o] = R.pos; flag[o] = (uint16_t)R.flag; seq_len[o] = (uint16_t)R.seq; chr[o] = R.chr;
        seq_off[o] = S.base[1] + wb[1] + incl[1] - R.seq;
        cigar_off[o] = S.base[2] + wb[2] + incl[2] - R.cig;
        if (!derive) md_off[o] = S.base[3] + wb[3] + incl[3] - R.md;
        src[o] = R.p; md_at[o] = R.md_at;
    }
    if (tile + 1u == n_tiles && tid == 0) {
        const uint64_t n = S.base[0] + tot[0];
        words[3] = n; words[4] = S.base[1] + tot[1]; words[5] = S.base[2] + tot[2]; words[6] = S.base[3] + tot[3];
        seq_off[n] = words[4]; cigar_off[n] = words[5];
        if (!derive) md_off[n] = words[6];
    }
}

/* a thread per read: SEQ, CIGAR and MD text; chromosome runs as (first read | chromosome << 32, its POS) and (last read, its
   POS) pairs, each list in any order */
__global__ void k10_write_kernel(const uint8_t *__restrict__ s, uint64_t n, uint32_t derive, const uint64_t *__restrict__ src,
                                 const uint64_t *__restrict__ md_at, const uint32_t *__restrict__ chr, const uint32_t *__restrict__ pos,
                                 const uint64_t *__restrict__ seq_off,
                                 const uint64_t *__restrict__ cigar_off, const uint64_t *__restrict__ md_off, uint8_t *seq, uint8_t *cigar,
                                 uint8_t *md, uint64_t *run_first, uint64_t *run_last, uint64_t *words) {
    const uint64_t o = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n) return;
    const uint64_t p = src[o];
    const uint32_t lrn = s[p + 12], n_cig = k10_u16(s, p + 16), l_seq = k10_u32(s, p + 20);
    const uint64_t c0 = p + 36u + lrn, s0 = c0 + 4ull * n_cig;
    uint8_t *d = seq + seq_off[o];
    for (uint32_t j = 0; j < l_seq; j++) d[j] = "=ACMGRSVTWYHKDBN"[(s[s0 + (j >> 1)] >> ((~j & 1u) * 4u)) & 15u];
    uint8_t *c = cigar + cigar_off[o];
    if (!n_cig) *c = '*';
    for (uint32_t k = 0; k < n_cig; k++) {
        const uint32_t v = k10_u32(s, c0 + 4ull * k);
        uint32_t len = v >> 4;
        const uint32_t nd = k10_digits(len);
        for (uint32_t i = nd; i-- > 0;) { c[i] = (uint8_t)('0' + len % 10u); len /= 10u; }
        c[nd] = (uint8_t)"MIDNSHP=X"[v & 15u];
        c += nd + 1u;
    }
    if (!derive) {
        const uint64_t a = md_at[o], l = md_off[o + 1] - md_off[o];
        uint8_t *m = md + md_off[o];
        for (uint64_t j = 0; j < l; j++) m[j] = s[a + j];
    }
    const uint32_t ch = chr[o];
    if (o == 0 || chr[o - 1] != ch) {
        const uint64_t i = atomicAdd(reinterpret_cast<unsigned long long *>(&words[7]), 1ull);
        run_first[2 * i] = o << 32 >> 32 | (uint64_t)ch << 32;   /* read ordinal < 2^32 (cbcg_batch's limit) */
        run_first[2 * i + 1] = pos[o];
    }
    if (o + 1 == n || chr[o + 1] != ch) {
        const uint64_t i = atomicAdd(reinterpret_cast<unsigned long long *>(&words[8]), 1ull);
        run_last[2 * i] = o; run_last[2 * i + 1] = pos[o];
    }
}

uint64_t bam_in_num_tiles(uint64_t n_records) { return (n_records + K10_TILE - 1u) / K10_TILE; }

int launch_bam_count(const uint8_t *stream, const uint64_t *rec_start, uint64_t n_rec, const int32_t *map, int32_t n_ref, uint32_t derive,
                     const DevBatch &b, uint64_t *src, uint64_t *md_at, uint64_t *tile_desc, uint32_t *ticket, uint64_t *words, uint32_t *lens,
                     unsigned long long *err, cudaStream_t st) {
    if (!n_rec) return 0;
    const uint64_t tiles = bam_in_num_tiles(n_rec);
    if (cudaMemsetAsync(tile_desc, 0, 4u * tiles * sizeof(uint64_t), st) != cudaSuccess) return -1;
    if (cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st) != cudaSuccess) return -1;
    k10_count_kernel<<<(unsigned)tiles, K10_TILE, 0, st>>>(stream, rec_start, n_rec, map, n_ref, derive, const_cast<uint32_t *>(b.pos),
                                                           const_cast<uint16_t *>(b.flag), const_cast<uint16_t *>(b.seq_len),
                                                           const_cast<uint32_t *>(b.chr), const_cast<uint64_t *>(b.seq_off),
                                                           const_cast<uint64_t *>(b.cigar_off), const_cast<uint64_t *>(b.md_off), src, md_at,
                                                           tile_desc, ticket, words, lens, err);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_bam_write(const uint8_t *stream, const DevBatch &b, uint32_t derive, const uint64_t *src, const uint64_t *md_at, uint64_t *run_first,
                     uint64_t *run_last, uint64_t *words, cudaStream_t st) {
    if (!b.n_reads) return 0;
    k10_write_kernel<<<(unsigned)((b.n_reads + 255u) / 256u), 256, 0, st>>>(stream, b.n_reads, derive, src, md_at, b.chr, b.pos, b.seq_off, b.cigar_off,
                                                                            b.md_off, const_cast<uint8_t *>(b.seq), const_cast<uint8_t *>(b.cigar),
                                                                            const_cast<uint8_t *>(b.md), run_first, run_last, words);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
