/*
 * api.cu -- the C ABI of include/cbcg.h over the K1 / K2 / K3 kernels.
 *
 * Host side of the drop-in boundary: owns every device buffer, sequences the kernels on one stream,
 * turns device error words into cbcg_status codes, and frames the blocked container ("CBCB": header,
 * per-block index, payload; the reference stream has no framing, src/compression.c:128-155). There is
 * no CPU coding path here: every entry point that codes, extracts or reconstructs launches kernels,
 * and cbcg_create fails without an sm_100 device.
 */
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "internal.h"
#include "container.h"

#define ABI_VERSION 1

/* ------------------------------------------------------------------------------------------------ */
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct ChrRun { uint64_t first, n; uint32_t chr; };
#define PIPE_MAX 6             /* side streams: with the main and the copy stream that makes 8, the default number of hardware queues (more would alias and serialise) */

/* small device words + their pinned host mirror */
struct Words {
    unsigned long long err;
    uint64_t total_edits;
    uint64_t total_bytes;
    uint64_t totals[5];
    uint32_t ticket;
    uint32_t pad;
    uint64_t chain[2];                        /* pipelined encode: edit entries so far, ping-pong between K1 launches */
    uint64_t n_selected;                      /* region decode: reads K5 kept */
    uint64_t md_chain[2];                     /* MD derivation (K7): MD bytes of the batch ([0]), or so far, ping-pong between chunk launches */
};

struct cbcg_ctx {
    int device = 0;
    cudaStream_t st = nullptr;
    cudaEvent_t ev[8] = {};
    cudaEvent_t kev[4] = {};                  /* tight around K1 (0,1) and K3 (2,3) */
    cudaEvent_t mark[4] = {};
    /* pipelined host-buffer calls (cbcg_encode / cbcg_decode on large batches): a copy stream, side streams for the
       groups of last-generation blocks, and the events that order them */
    cudaStream_t cs = nullptr, ps[PIPE_MAX] = {};
    cudaStream_t hp = nullptr;                /* high priority: the early generations of a resident encode, beside K1 on a side stream */
    cudaEvent_t cev[PIPE_MAX + 2] = {}, kev2[PIPE_MAX + 2] = {}, dev2[PIPE_MAX + 2] = {}, tev[2 * PIPE_MAX + 4] = {};
    bool pipe_ready = false;
    char errtext[512] = {0};
    cbcg_stats stats = {};

    /* genome */
    DevBuf g_bases, g_off, g_len, g_names;
    std::vector<std::string> names;
    std::vector<uint64_t> h_off, h_len;
    DevGenome dg = {};

    /* resident batch */
    DevBuf b_pos, b_flag, b_len, b_chr, b_soff, b_seq, b_coff, b_cigar, b_moff, b_md;
    DevBatch db = {};
    std::vector<ChrRun> runs;
    uint64_t total_bases = 0;
    bool have_batch = false;
    bool batch_no_md = false;                 /* the resident batch came without MD: K7 derives it (DESIGN.md 5d) */

    /* compact batches (cbcg_batch_compact): staging for what is unpacked on the device */
    DevBuf c_seq2, c_cl, c_ml, c_tile, c_rfirst, c_rchr, c_er, c_eb, c_ec;
    uint64_t *h_tile = nullptr; size_t h_tile_cap = 0;   /* pinned: one (seq, seq2, cigar, md) byte offset per tile of 128 reads */

    /* work buffers */
    DevBuf recs, edits, chr_out, tile_desc, words, blocks, ws, scratch, payload, out_off, symbols, seq_out;
    DevBuf cig_cls, cig_exc, cig_out;          /* CIGAR recovery (k4_cigar.cu): classes, verbatim texts, emitted text */
    DevBuf tri;                                /* two-kernel encode: the symbols' intervals between the model and the interval kernel */
    DevBuf reg, sel_recs, sel_chr, sel_ids;    /* region decode (k5_region.cu): intervals + ordinal runs, and the kept reads */
    DevBuf sam_aux, sam_out;                   /* SAM output (k6_sam.cu): name lengths, CIGAR classes and texts; the text */
    DevBuf snap_a, snap_b, fin;                /* generation snapshots and per-block final states (gen_mode 1) */
    std::vector<std::pair<uint32_t, uint32_t>> gens;   /* (first block, block count) per generation of the last cut */
    uint32_t layout = 1;                       /* the call in progress: 1 = one stream per block, 4 = four substreams, 0 = four in the narrow early generations */
    uint32_t layout_mode = 0;                  /* the same as container mode bits (CBCG_MODE_SPLIT4 / split generations), set by the cut or read from the header */
    uint32_t max_block_reads = 0;              /* longest block of the last cut / index: sets the merged snapshots' FLAG total (cbcg_flag_target) */
    Words *hw = nullptr;                       /* pinned */
    BlockDesc *hblocks = nullptr; size_t hblocks_cap = 0;   /* pinned */

    /* result of the last encode */
    bool have_encoded = false;
    uint32_t enc_L = 0, enc_block_reads = 0, enc_gen_mode = 0, enc_legacy = 0, enc_max_len = 0, enc_fixed = 0, enc_layout_mode = 0;
    uint32_t batch_min_len = 0;               /* shortest read of the resident batch (host scan at upload) */
    bool batch_indel_heavy = false;           /* CIGAR text per read well beyond "<len>M": most reads carry indels / clips (picks the model kernel's edit walk) */
    uint64_t enc_n_reads = 0, enc_n_edits = 0, enc_n_blocks = 0, enc_payload_bytes = 0;
    std::vector<uint8_t> enc_head;             /* container header + index */

    /* result of the last decode */
    bool have_decoded = false;
    uint64_t dec_bytes = 0, dec_n_reads = 0;
};

static int fail(cbcg_ctx *c, int status, const char *fmt, ...) {
    if (c) {
        va_list ap; va_start(ap, fmt);
        vsnprintf(c->errtext, sizeof c->errtext, fmt, ap);
        va_end(ap);
    }
    return status;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) \
    return fail(ctx, e_ == cudaErrorMemoryAllocation ? CBCG_ERR_NOMEM : CBCG_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
#define TRY(call) do { int r_ = (call); if (r_) return r_; } while (0)

static int ensure(cbcg_ctx *ctx, DevBuf &b, size_t bytes) {
    bytes = (bytes + 255u) & ~(size_t)255u;
    if (bytes <= b.cap && b.p) return 0;
    if (b.p) { CU(cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 4096;            /* a little slack so near-equal batches do not reallocate */
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) { want = bytes; (void)cudaGetLastError(); e = cudaMalloc(&b.p, want); }
    if (e != cudaSuccess) { b.p = nullptr; (void)cudaGetLastError(); return fail(ctx, CBCG_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); }
    b.cap = want;
    return 0;
}
static int ensure_hblocks(cbcg_ctx *ctx, size_t n) {
    if (n <= ctx->hblocks_cap) return 0;
    if (ctx->hblocks) cudaFreeHost(ctx->hblocks);
    ctx->hblocks = nullptr; ctx->hblocks_cap = 0;
    size_t want = n + n / 4 + 64;
    CU(cudaMallocHost(&ctx->hblocks, want * sizeof(BlockDesc)));
    ctx->hblocks_cap = want;
    return 0;
}
static void free_buf(DevBuf &b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }

/* device words */
#define W_OFF(field) (offsetof(Words, field))
template <class T> static T *wptr(cbcg_ctx *ctx, size_t off) { return reinterpret_cast<T *>(ctx->words.as<uint8_t>() + off); }

static int device_error(cbcg_ctx *ctx, const char *stage) {
    const unsigned long long v = ctx->hw->err;
    if (!v) return 0;
    const int code = -(int)(v >> 40);
    const unsigned long long item = v & 0xffffffffffull;
    return fail(ctx, code, "%s: %s at item %llu", stage, cbcg_strerror(code), item);
}

/* ------------------------------------------------------------------------------------------------ lifetime */
extern "C" int cbcg_abi_version(void) { return ABI_VERSION; }

extern "C" const char *cbcg_strerror(int s) {
    switch (s) {
        case CBCG_OK: return "ok";
        case CBCG_ERR_ARG: return "bad argument";
        case CBCG_ERR_CUDA: return "CUDA runtime error";
        case CBCG_ERR_NO_DEVICE: return "no usable sm_100 GPU (there is no CPU path)";
        case CBCG_ERR_NOMEM: return "out of memory";
        case CBCG_ERR_CAPACITY: return "output buffer too small";
        case CBCG_ERR_INPUT: return "read outside what the reference can code";
        case CBCG_ERR_NO_REFERENCE: return "reference genome missing or chromosome out of range";
        case CBCG_ERR_FORMAT: return "malformed container";
        case CBCG_ERR_CORRUPT: return "corrupt bitstream";
        case CBCG_ERR_LIMIT: return "internal table limit reached";
        case CBCG_ERR_INTERNAL: return "internal error";
        default: return "unknown status";
    }
}

extern "C" const char *cbcg_last_error(const cbcg_ctx *ctx) { return ctx ? ctx->errtext : "no context"; }

extern "C" int cbcg_create(int device, cbcg_ctx **out) {
    if (!out) return CBCG_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) { (void)cudaGetLastError(); return CBCG_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return CBCG_ERR_NO_DEVICE;
    if (prop.major != 10) return CBCG_ERR_NO_DEVICE;     /* kernels are sm_100a only */
    if (cudaSetDevice(device) != cudaSuccess) return CBCG_ERR_NO_DEVICE;
    cbcg_ctx *ctx = new (std::nothrow) cbcg_ctx();
    if (!ctx) return CBCG_ERR_NOMEM;
    ctx->device = device;
    if (cudaStreamCreateWithFlags(&ctx->st, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return CBCG_ERR_CUDA; }
    for (auto &e : ctx->ev) if (cudaEventCreate(&e) != cudaSuccess) { delete ctx; return CBCG_ERR_CUDA; }
    for (auto &e : ctx->mark) if (cudaEventCreate(&e) != cudaSuccess) { delete ctx; return CBCG_ERR_CUDA; }
    for (auto &e : ctx->kev) if (cudaEventCreate(&e) != cudaSuccess) { delete ctx; return CBCG_ERR_CUDA; }
    if (cudaMallocHost(&ctx->hw, sizeof(Words)) != cudaSuccess) { delete ctx; return CBCG_ERR_NOMEM; }
    memset(ctx->hw, 0, sizeof(Words));
    if (ensure(ctx, ctx->words, sizeof(Words))) { cudaFreeHost(ctx->hw); delete ctx; return CBCG_ERR_NOMEM; }
    cudaMemsetAsync(ctx->words.p, 0, sizeof(Words), ctx->st);
    cudaStreamSynchronize(ctx->st);
    *out = ctx;
    return CBCG_OK;
}

extern "C" void cbcg_destroy(cbcg_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->st) cudaStreamSynchronize(ctx->st);
    DevBuf *all[] = { &ctx->g_bases, &ctx->g_off, &ctx->g_len, &ctx->g_names, &ctx->b_pos, &ctx->b_flag, &ctx->b_len, &ctx->b_chr,
                      &ctx->b_soff, &ctx->b_seq, &ctx->b_coff, &ctx->b_cigar, &ctx->b_moff, &ctx->b_md, &ctx->recs, &ctx->edits,
                      &ctx->chr_out, &ctx->tile_desc, &ctx->words, &ctx->blocks, &ctx->ws, &ctx->scratch, &ctx->payload,
                      &ctx->out_off, &ctx->symbols, &ctx->seq_out, &ctx->snap_a, &ctx->snap_b, &ctx->fin, &ctx->cig_cls, &ctx->cig_exc, &ctx->cig_out };
    for (DevBuf *b : all) free_buf(*b);
    if (ctx->hw) cudaFreeHost(ctx->hw);
    if (ctx->hblocks) cudaFreeHost(ctx->hblocks);
    if (ctx->h_tile) cudaFreeHost(ctx->h_tile);
    for (DevBuf *d : { &ctx->c_seq2, &ctx->c_cl, &ctx->c_ml, &ctx->c_tile, &ctx->c_rfirst, &ctx->c_rchr, &ctx->c_er, &ctx->c_eb, &ctx->c_ec,
                       &ctx->reg, &ctx->sel_recs, &ctx->sel_chr, &ctx->sel_ids, &ctx->sam_aux, &ctx->sam_out }) free_buf(*d);
    for (auto &e : ctx->ev) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->mark) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->kev) if (e) cudaEventDestroy(e);
    if (ctx->st) cudaStreamDestroy(ctx->st);
    if (ctx->cs) cudaStreamDestroy(ctx->cs);
    if (ctx->hp) cudaStreamDestroy(ctx->hp);
    for (auto &s : ctx->ps) if (s) cudaStreamDestroy(s);
    for (auto &e : ctx->cev) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->kev2) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->dev2) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->tev) if (e) cudaEventDestroy(e);
    delete ctx;
}

extern "C" int cbcg_get_stats(const cbcg_ctx *ctx, cbcg_stats *out) {
    if (!ctx || !out) return CBCG_ERR_ARG;
    *out = ctx->stats;
    return CBCG_OK;
}

/* Timing marks on the library's own stream (torch events only see torch's stream). */
extern "C" int cbcg_mark(cbcg_ctx *ctx, int slot) {
    if (!ctx || slot < 0 || slot >= 4) return fail(ctx, CBCG_ERR_ARG, "cbcg_mark: bad slot");
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventRecord(ctx->mark[slot], ctx->st));
    return CBCG_OK;
}
extern "C" int cbcg_elapsed_ms(cbcg_ctx *ctx, int from, int to, float *ms) {
    if (!ctx || !ms || from < 0 || from >= 4 || to < 0 || to >= 4) return fail(ctx, CBCG_ERR_ARG, "cbcg_elapsed_ms: bad argument");
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventSynchronize(ctx->mark[to]));
    CU(cudaEventElapsedTime(ms, ctx->mark[from], ctx->mark[to]));
    return CBCG_OK;
}

extern "C" void *cbcg_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void cbcg_host_free(void *p) { if (p) cudaFreeHost(p); }

/* ------------------------------------------------------------------------------------------------ genome */
__global__ void genome_prepare_kernel(uint8_t *bases, uint64_t off, uint64_t len, uint64_t span) {
    /* upper-case the record (store_reference_in_memory, src/read_decompression.c:38-44) and fill its tail pad */
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < span; i += stride) {
        uint8_t c = (i < len) ? bases[off + i] : (uint8_t)'N';
        if (c >= 'a' && c <= 'z') c = (uint8_t)(c - 32);
        bases[off + i] = c;
    }
}

extern "C" int cbcg_set_reference(cbcg_ctx *ctx, uint32_t n_chr, const char *const *names,
                                  const uint8_t *const *bases, const uint64_t *len) {
    if (!ctx || !n_chr || !bases || !len || n_chr > MAX_CHR) return fail(ctx, CBCG_ERR_ARG, "cbcg_set_reference: bad argument");
    CU(cudaSetDevice(ctx->device));
    ctx->names.clear(); ctx->h_off.clear(); ctx->h_len.clear();
    uint64_t total = 0;
    for (uint32_t c = 0; c < n_chr; c++) {
        if (!bases[c]) return fail(ctx, CBCG_ERR_ARG, "cbcg_set_reference: NULL record %u", c);
        char tmp[32];
        const char *nm = (names && names[c]) ? names[c] : (snprintf(tmp, sizeof tmp, "chr%u", c + 1), tmp);
        if (strlen(nm) >= MAX_NAME) return fail(ctx, CBCG_ERR_ARG, "chromosome name too long");
        ctx->names.push_back(nm);
        ctx->h_off.push_back(total);
        ctx->h_len.push_back(len[c]);
        total += (len[c] + REF_PAD + 255u) & ~255ull;
    }
    TRY(ensure(ctx, ctx->g_bases, total + 256));
    TRY(ensure(ctx, ctx->g_off, n_chr * 8));
    TRY(ensure(ctx, ctx->g_len, n_chr * 8));
    TRY(ensure(ctx, ctx->g_names, (size_t)n_chr * MAX_NAME));
    std::vector<uint8_t> nm((size_t)n_chr * MAX_NAME, 0);
    for (uint32_t c = 0; c < n_chr; c++) memcpy(&nm[(size_t)c * MAX_NAME], ctx->names[c].c_str(), ctx->names[c].size());
    CU(cudaMemcpyAsync(ctx->g_off.p, ctx->h_off.data(), n_chr * 8, cudaMemcpyHostToDevice, ctx->st));
    CU(cudaMemcpyAsync(ctx->g_len.p, ctx->h_len.data(), n_chr * 8, cudaMemcpyHostToDevice, ctx->st));
    CU(cudaMemcpyAsync(ctx->g_names.p, nm.data(), nm.size(), cudaMemcpyHostToDevice, ctx->st));
    for (uint32_t c = 0; c < n_chr; c++) {
        if (len[c]) CU(cudaMemcpyAsync(ctx->g_bases.as<uint8_t>() + ctx->h_off[c], bases[c], len[c], cudaMemcpyHostToDevice, ctx->st));
        const uint64_t span = (len[c] + REF_PAD + 255u) & ~255ull;
        genome_prepare_kernel<<<(unsigned)std::min<uint64_t>(148u * 8u, (span + 255u) / 256u), 256, 0, ctx->st>>>(
            ctx->g_bases.as<uint8_t>(), ctx->h_off[c], len[c], span);
    }
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->st));
    ctx->dg.n_chr = n_chr;
    ctx->dg.bases = ctx->g_bases.as<uint8_t>();
    ctx->dg.chr_off = ctx->g_off.as<uint64_t>();
    ctx->dg.chr_len = ctx->g_len.as<uint64_t>();
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ batch */
static int check_batch(cbcg_ctx *ctx, const cbcg_batch *b) {
    if (!b) return fail(ctx, CBCG_ERR_ARG, "NULL batch");
    if (b->n_reads == 0) return 0;
    const bool no_md = !b->md_off && !b->md;               /* no MD: K7 derives it */
    if (!b->pos || !b->flag || !b->seq_len || !b->chr || !b->seq_off || !b->seq || !b->cigar_off || !b->cigar || (!no_md && (!b->md_off || !b->md)))
        return fail(ctx, CBCG_ERR_ARG, "batch has NULL arrays");
    if (b->n_reads >= 0xfffffff0ull) return fail(ctx, CBCG_ERR_ARG, "more than 2^32 reads in one shard");
    const uint64_t n = b->n_reads;                          /* the copies are sized from the pool offsets' end points */
    if (b->seq_off[n] < b->seq_off[0] || b->cigar_off[n] < b->cigar_off[0] || (!no_md && b->md_off[n] < b->md_off[0]))
        return fail(ctx, CBCG_ERR_INPUT, "batch pool offsets decrease");
    return 0;
}

/* MD pool of a batch without MD, before K7 has counted it: canonical MD is about a digit or two per run of matches and two
 * or three bytes per edit, so an eighth of the bases plus 8 per read covers a batch with one edit in twenty bases several
 * times over. A batch that needs more is derived again at the exact size (derive_md). */
static uint64_t md_bytes_guess(uint64_t bases, uint64_t n) { return bases / 8 + 8 * n + 4096; }

/* Device buffers for the batch and ctx->db pointing at them (no copies yet). */
static int batch_prepare(cbcg_ctx *ctx, const cbcg_batch *b) {
    const uint64_t n = b->n_reads;
    ctx->have_batch = false; ctx->have_encoded = false;
    ctx->batch_no_md = !b->md_off;
    ctx->runs.clear();
    ctx->stats = cbcg_stats();
    if (n) {
        const uint64_t seq_b = b->seq_off[n], cig_b = b->cigar_off[n], md_b = b->md_off ? b->md_off[n] : md_bytes_guess(seq_b - b->seq_off[0], n);
        TRY(ensure(ctx, ctx->b_pos, n * 4));  TRY(ensure(ctx, ctx->b_flag, n * 2)); TRY(ensure(ctx, ctx->b_len, n * 2));
        TRY(ensure(ctx, ctx->b_chr, n * 4));
        TRY(ensure(ctx, ctx->b_soff, (n + 1) * 8)); TRY(ensure(ctx, ctx->b_coff, (n + 1) * 8)); TRY(ensure(ctx, ctx->b_moff, (n + 1) * 8));
        TRY(ensure(ctx, ctx->b_seq, seq_b + POOL_PAD)); TRY(ensure(ctx, ctx->b_cigar, cig_b + POOL_PAD)); TRY(ensure(ctx, ctx->b_md, md_b + POOL_PAD));
    }
    ctx->db.n_reads = n;
    ctx->db.pos = ctx->b_pos.as<uint32_t>(); ctx->db.flag = ctx->b_flag.as<uint16_t>(); ctx->db.seq_len = ctx->b_len.as<uint16_t>();
    ctx->db.chr = ctx->b_chr.as<uint32_t>();
    ctx->db.seq_off = ctx->b_soff.as<uint64_t>(); ctx->db.seq = ctx->b_seq.as<uint8_t>();
    ctx->db.cigar_off = ctx->b_coff.as<uint64_t>(); ctx->db.cigar = ctx->b_cigar.as<uint8_t>();
    ctx->db.md_off = ctx->b_moff.as<uint64_t>(); ctx->db.md = ctx->b_md.as<uint8_t>();
    return 0;
}
/* Reads [r0, r1) of every array of the batch, host -> device, on stream st (pool offsets are absolute, so a slice
   of the offset arrays indexes the same pools). */
static int batch_copy_range(cbcg_ctx *ctx, const cbcg_batch *b, uint64_t r0, uint64_t r1, cudaStream_t st, uint64_t *bytes) {
    if (r1 <= r0) return 0;
    const uint64_t m = r1 - r0;
    const bool md = b->md_off != nullptr;                   /* without MD there is none to copy: K7 writes md_off and the pool */
    const uint64_t s0 = b->seq_off[r0], s1 = b->seq_off[r1], c0 = b->cigar_off[r0], c1 = b->cigar_off[r1], m0 = md ? b->md_off[r0] : 0, m1 = md ? b->md_off[r1] : 0;
    struct { void *d; const void *h; uint64_t bytes; } cp[] = {
        { ctx->b_pos.as<uint32_t>() + r0, b->pos + r0, m * 4 }, { ctx->b_flag.as<uint16_t>() + r0, b->flag + r0, m * 2 },
        { ctx->b_len.as<uint16_t>() + r0, b->seq_len + r0, m * 2 }, { ctx->b_chr.as<uint32_t>() + r0, b->chr + r0, m * 4 },
        { ctx->b_soff.as<uint64_t>() + r0, b->seq_off + r0, (m + 1) * 8 }, { ctx->b_coff.as<uint64_t>() + r0, b->cigar_off + r0, (m + 1) * 8 },
        { ctx->b_moff.as<uint64_t>() + r0, md ? b->md_off + r0 : nullptr, md ? (m + 1) * 8 : 0 }, { ctx->b_seq.as<uint8_t>() + s0, b->seq + s0, s1 - s0 },
        { ctx->b_cigar.as<uint8_t>() + c0, b->cigar + c0, c1 - c0 }, { ctx->b_md.as<uint8_t>() + m0, md ? b->md + m0 : nullptr, m1 - m0 } };
    for (auto &c : cp) { if (c.bytes) CU(cudaMemcpyAsync(c.d, c.h, c.bytes, cudaMemcpyHostToDevice, st)); *bytes += c.bytes; }
    return 0;
}
/* K1's reference window (DevBatch.ref_cap): bytes of reference that 128 position-adjacent reads span at this batch's
 * coverage, twice over, plus a read. From the first and last POS of every chromosome run. */
static uint32_t ref_window_estimate(const cbcg_ctx *ctx, const uint32_t *pos, uint64_t n, uint32_t max_len) {
    if (!n || !pos) return 0u;
    uint64_t span = 0;
    for (const ChrRun &r : ctx->runs) if (r.n) { const uint32_t a = pos[r.first], z = pos[r.first + r.n - 1]; if (z > a) span += z - a; }
    const double per_read = (double)span / (double)n;
    const double want = per_read * 128.0 * 2.0 + max_len + 64.0;
    return want > 1e9 ? 0u : (uint32_t)want;
}
/* Host scan of the batch: chromosome runs (blocks never span chromosomes), longest and shortest read. */
static int batch_scan(cbcg_ctx *ctx, const cbcg_batch *b) {
    const uint64_t n = b->n_reads;
    uint32_t max_len = 0, min_len = 0xffffffffu;
    ctx->runs.clear();
    uint64_t bad = 0;
    if (n) {
        const uint16_t *sl = b->seq_len;
        const uint64_t *so = b->seq_off, *co = b->cigar_off, *mo = b->md_off ? b->md_off : b->cigar_off;   /* no MD: nothing more to check */
        for (uint64_t r = 0; r < n; r++) {
            const uint32_t l = sl[r]; max_len = l > max_len ? l : max_len; min_len = l < min_len ? l : min_len;
            /* SEQ pool entries are exactly the reads; CIGAR / MD offsets never decrease (kernels size their loops from them) */
            bad |= (so[r + 1] - so[r]) ^ (uint64_t)l;
            bad |= (uint64_t)(co[r + 1] < co[r]) | (uint64_t)(mo[r + 1] < mo[r]);
        }
        ChrRun run = { 0, 0, b->chr[0] };
        const uint32_t *ch = b->chr;
        for (uint64_t r = 0; r < n; r++) {
            if (ch[r] != run.chr) { ctx->runs.push_back(run); run.first = r; run.n = 0; run.chr = ch[r]; }
            run.n++;
        }
        ctx->runs.push_back(run);
    }
    ctx->db.max_len = max_len;
    ctx->db.ref_cap = ref_window_estimate(ctx, b->pos, n, max_len);
    ctx->batch_indel_heavy = n && (b->cigar_off[n] - b->cigar_off[0]) > n * 6ull;      /* "150M" is 4 bytes, "60M1I39M" 8 */
    ctx->batch_min_len = n ? min_len : 0;
    ctx->total_bases = n ? b->seq_off[n] - b->seq_off[0] : 0;
    if (n && (min_len == 0 || max_len > CBCG_MAX_READ_LEN))
        return fail(ctx, CBCG_ERR_INPUT, "read length outside 1..%u (shortest %u, longest %u)", CBCG_MAX_READ_LEN, min_len, max_len);
    if (bad) return fail(ctx, CBCG_ERR_INPUT, "batch offsets inconsistent: seq_off must advance by seq_len, cigar_off / md_off must not decrease");
    return 0;
}

static int reset_words(cbcg_ctx *ctx);
static int fetch_words(cbcg_ctx *ctx);
static int derive_md(cbcg_ctx *ctx, uint64_t need);
/* ---- compact batches: what crosses the link packed, rebuilt into the layout above on the device (k0_unpack.cu) */
struct BatchSrc { const cbcg_batch *full; const cbcg_batch_compact *compact; uint64_t n; };
static int check_compact(cbcg_ctx *ctx, const cbcg_batch_compact *b) {
    if (!b) return fail(ctx, CBCG_ERR_ARG, "NULL batch");
    if (b->n_reads == 0) return 0;
    const bool no_md = !b->md_len && !b->md;               /* no MD: K7 derives it */
    if (!b->pos || !b->flag || !b->seq_len || !b->cigar_len || (!no_md && (!b->md_len || !b->md)) || !b->n_runs || !b->run_first || !b->run_chr || !b->seq2 || !b->cigar ||
        !b->tile_base || (b->n_exc && (!b->exc_read || !b->exc_base || !b->exc_char)))
        return fail(ctx, CBCG_ERR_ARG, "compact batch has NULL arrays");
    if (b->n_reads >= 0xfffffff0ull) return fail(ctx, CBCG_ERR_ARG, "more than 2^32 reads in one shard");
    if (b->run_first[0] != 0) return fail(ctx, CBCG_ERR_INPUT, "the first chromosome run must start at read 0");
    if (b->min_len == 0 || b->max_len > CBCG_MAX_READ_LEN || b->min_len > b->max_len)
        return fail(ctx, CBCG_ERR_INPUT, "read length outside 1..%u (shortest %u, longest %u)", CBCG_MAX_READ_LEN, b->min_len, b->max_len);
    const uint64_t tiles = (b->n_reads + 127u) / 128u;
    for (int q = 0; q < 4; q++) if (b->tile_base[q] != 0) return fail(ctx, CBCG_ERR_INPUT, "compact batch: tile offsets must start at 0");
    if (b->tile_base[tiles * 4] > b->n_reads * (uint64_t)b->max_len || b->tile_base[tiles * 4 + 1] > b->tile_base[tiles * 4])
        return fail(ctx, CBCG_ERR_INPUT, "compact batch: totals inconsistent");
    if (no_md)
        for (uint64_t t = 0; t <= tiles; t++) if (b->tile_base[t * 4 + 3]) return fail(ctx, CBCG_ERR_INPUT, "compact batch without MD: its tile offsets count MD bytes");
    return 0;
}
/* Device buffers of a compact batch and ctx->db; chromosome runs and the exception list are checked here (both short),
 * the per-read lengths are checked against the tile offsets by the unpack kernel. No pass over the reads on the host. */
static int compact_buffers(cbcg_ctx *ctx, const cbcg_batch_compact *b) {
    const uint64_t n = b->n_reads, tiles = (n + 127u) / 128u;
    ctx->have_batch = false; ctx->have_encoded = false;
    ctx->batch_no_md = !b->md_len;
    ctx->runs.clear();
    ctx->stats = cbcg_stats();
    uint64_t seq_b = 0;
    if (n) {
        for (uint64_t t = 0; t < tiles; t++)
            for (int q = 0; q < 4; q++) if (b->tile_base[(t + 1) * 4 + q] < b->tile_base[t * 4 + q]) return fail(ctx, CBCG_ERR_INPUT, "compact batch: tile offsets decrease");
        for (uint32_t k = 0; k < b->n_runs; k++) {
            const uint64_t first = b->run_first[k], end = k + 1 < b->n_runs ? b->run_first[k + 1] : n;
            if (end <= first || end > n) return fail(ctx, CBCG_ERR_INPUT, "compact batch: chromosome runs out of order");
            ctx->runs.push_back({ first, end - first, b->run_chr[k] });
        }
        for (uint64_t e = 1; e < b->n_exc; e++) if (b->exc_read[e] < b->exc_read[e - 1]) return fail(ctx, CBCG_ERR_INPUT, "compact batch: exception list not sorted by read");
        if (b->n_exc && b->exc_read[b->n_exc - 1] >= n) return fail(ctx, CBCG_ERR_INPUT, "compact batch: exception outside the batch");
        for (uint64_t e = 0; e < b->n_exc; e++) if (b->exc_base[e] >= b->max_len) return fail(ctx, CBCG_ERR_INPUT, "compact batch: exception beyond the longest read");
        const uint64_t *tot = b->tile_base + tiles * 4;
        seq_b = tot[0];
        const uint64_t s2_b = tot[1], cig_b = tot[2], md_b = b->md_len ? tot[3] : md_bytes_guess(seq_b, n);
        TRY(ensure(ctx, ctx->b_pos, n * 4));  TRY(ensure(ctx, ctx->b_flag, n * 2)); TRY(ensure(ctx, ctx->b_len, n * 2));
        TRY(ensure(ctx, ctx->b_chr, n * 4));
        TRY(ensure(ctx, ctx->b_soff, (n + 1) * 8)); TRY(ensure(ctx, ctx->b_coff, (n + 1) * 8)); TRY(ensure(ctx, ctx->b_moff, (n + 1) * 8));
        TRY(ensure(ctx, ctx->b_seq, seq_b + 4 * 0u + POOL_PAD)); TRY(ensure(ctx, ctx->b_cigar, cig_b + POOL_PAD)); TRY(ensure(ctx, ctx->b_md, md_b + POOL_PAD));
        TRY(ensure(ctx, ctx->c_seq2, s2_b + POOL_PAD)); TRY(ensure(ctx, ctx->c_cl, n * 2)); TRY(ensure(ctx, ctx->c_ml, n * 2));
        TRY(ensure(ctx, ctx->c_tile, (tiles + 1) * 32)); TRY(ensure(ctx, ctx->c_rfirst, (uint64_t)b->n_runs * 8)); TRY(ensure(ctx, ctx->c_rchr, (uint64_t)b->n_runs * 4));
        TRY(ensure(ctx, ctx->c_er, b->n_exc * 4 + 16)); TRY(ensure(ctx, ctx->c_eb, b->n_exc * 2 + 16)); TRY(ensure(ctx, ctx->c_ec, b->n_exc + 16));
    }
    ctx->db.n_reads = n;
    ctx->db.pos = ctx->b_pos.as<uint32_t>(); ctx->db.flag = ctx->b_flag.as<uint16_t>(); ctx->db.seq_len = ctx->b_len.as<uint16_t>();
    ctx->db.chr = ctx->b_chr.as<uint32_t>();
    ctx->db.seq_off = ctx->b_soff.as<uint64_t>(); ctx->db.seq = ctx->b_seq.as<uint8_t>();
    ctx->db.cigar_off = ctx->b_coff.as<uint64_t>(); ctx->db.cigar = ctx->b_cigar.as<uint8_t>();
    ctx->db.md_off = ctx->b_moff.as<uint64_t>(); ctx->db.md = ctx->b_md.as<uint8_t>();
    ctx->db.max_len = n ? b->max_len : 0; ctx->batch_min_len = n ? b->min_len : 0; ctx->total_bases = seq_b;
    ctx->db.ref_cap = ref_window_estimate(ctx, b->pos, n, ctx->db.max_len);
    ctx->batch_indel_heavy = n && b->tile_base[((n + 127) / 128) * 4 + 2] > n * 6ull;     /* CIGAR bytes of the whole batch */
    return 0;
}
/* the small pieces every chunk needs: tile offsets, chromosome runs, the exception list (first on the link) */
static int compact_copy_head(cbcg_ctx *ctx, const cbcg_batch_compact *b, cudaStream_t st, uint64_t *bytes) {
    const uint64_t tiles = (b->n_reads + 127u) / 128u;
    struct { void *d; const void *h; uint64_t bytes; } cp[] = {
        { ctx->c_tile.p, b->tile_base, (tiles + 1) * 32 }, { ctx->c_rfirst.p, b->run_first, (uint64_t)b->n_runs * 8 }, { ctx->c_rchr.p, b->run_chr, (uint64_t)b->n_runs * 4 },
        { ctx->c_er.p, b->exc_read, b->n_exc * 4 }, { ctx->c_eb.p, b->exc_base, b->n_exc * 2 }, { ctx->c_ec.p, b->exc_char, b->n_exc } };
    for (auto &c : cp) { if (c.bytes) CU(cudaMemcpyAsync(c.d, c.h, c.bytes, cudaMemcpyHostToDevice, st)); *bytes += c.bytes; }
    if (!b->md_len) CU(cudaMemsetAsync(ctx->c_ml.p, 0, b->n_reads * 2, st));   /* no MD: K0 lays out empty texts, K7 fills them in */
    return 0;
}
/* reads [r0, r1), both multiples of 128 (or the end of the batch) */
static int compact_copy_range(cbcg_ctx *ctx, const cbcg_batch_compact *b, uint64_t r0, uint64_t r1, cudaStream_t st, uint64_t *bytes) {
    if (r1 <= r0) return 0;
    const uint64_t m = r1 - r0;
    const uint64_t *t0 = b->tile_base + (r0 >> 7) * 4, *t1 = b->tile_base + ((r1 + 127u) >> 7) * 4;
    const uint64_t s0 = t0[1], s1 = t1[1], c0 = t0[2], c1 = t1[2], m0 = t0[3], m1 = t1[3];   /* no MD: m0 = m1 = 0 (check_compact) */
    struct { void *d; const void *h; uint64_t bytes; } cp[] = {
        { ctx->b_pos.as<uint32_t>() + r0, b->pos + r0, m * 4 }, { ctx->b_flag.as<uint16_t>() + r0, b->flag + r0, m * 2 },
        { ctx->b_len.as<uint16_t>() + r0, b->seq_len + r0, m * 2 }, { ctx->c_cl.as<uint16_t>() + r0, b->cigar_len + r0, m * 2 },
        { ctx->c_ml.as<uint16_t>() + r0, b->md_len ? b->md_len + r0 : nullptr, b->md_len ? m * 2 : 0 }, { ctx->c_seq2.as<uint8_t>() + s0, b->seq2 + s0, s1 - s0 },
        { ctx->b_cigar.as<uint8_t>() + c0, b->cigar + c0, c1 - c0 }, { ctx->b_md.as<uint8_t>() + m0, b->md ? b->md + m0 : nullptr, m1 - m0 } };
    for (auto &c : cp) { if (c.bytes) CU(cudaMemcpyAsync(c.d, c.h, c.bytes, cudaMemcpyHostToDevice, st)); *bytes += c.bytes; }
    return 0;
}
/* reads [r0, r1) (r0 a multiple of 128) from the staging buffers into the SoA batch */
static int compact_unpack_range(cbcg_ctx *ctx, const cbcg_batch_compact *b, uint64_t r0, uint64_t r1, cudaStream_t st) {
    if (r1 <= r0) return 0;
    if (launch_unpack(r0, r1, b->n_reads, ctx->b_len.as<uint16_t>(), ctx->c_cl.as<uint16_t>(), ctx->c_ml.as<uint16_t>(), ctx->c_seq2.as<uint8_t>(),
                      ctx->c_tile.as<uint64_t>(), ctx->c_rfirst.as<uint64_t>(), ctx->c_rchr.as<uint32_t>(), b->n_runs,
                      ctx->b_soff.as<uint64_t>(), ctx->b_coff.as<uint64_t>(), ctx->b_moff.as<uint64_t>(), ctx->b_seq.as<uint8_t>(), ctx->b_chr.as<uint32_t>(),
                      wptr<unsigned long long>(ctx, W_OFF(err)), st))
        return fail(ctx, CBCG_ERR_CUDA, "unpack launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    ctx->stats.kernel_launches++;
    if (b->n_exc) {
        const uint32_t *lo = std::lower_bound(b->exc_read, b->exc_read + b->n_exc, (uint32_t)r0);
        const uint32_t *hi = std::lower_bound(b->exc_read, b->exc_read + b->n_exc, (uint32_t)std::min<uint64_t>(r1, 0xffffffffull));
        const uint64_t e0 = (uint64_t)(lo - b->exc_read), e1 = (uint64_t)(hi - b->exc_read);
        if (e1 > e0) {
            if (launch_patch(ctx->c_er.as<uint32_t>() + e0, ctx->c_eb.as<uint16_t>() + e0, ctx->c_ec.as<uint8_t>() + e0, e1 - e0, ctx->b_soff.as<uint64_t>(), ctx->b_seq.as<uint8_t>(), st))
                return fail(ctx, CBCG_ERR_CUDA, "patch launch failed");
            ctx->stats.kernel_launches++;
        }
    }
    return 0;
}
static int src_prepare(cbcg_ctx *ctx, const BatchSrc &s) { return s.compact ? compact_buffers(ctx, s.compact) : batch_prepare(ctx, s.full); }
static int src_copy_range(cbcg_ctx *ctx, const BatchSrc &s, uint64_t r0, uint64_t r1, cudaStream_t st, uint64_t *bytes) {
    return s.compact ? compact_copy_range(ctx, s.compact, r0, r1, st, bytes) : batch_copy_range(ctx, s.full, r0, r1, st, bytes);
}

extern "C" int cbcg_batch_upload_compact(cbcg_ctx *ctx, const cbcg_batch_compact *b) {
    if (!ctx) return CBCG_ERR_ARG;
    TRY(check_compact(ctx, b));
    if (b->n_reads && !b->md_len && !ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "a batch without MD needs the reference: cbcg_set_reference has not been called");
    CU(cudaSetDevice(ctx->device));
    const uint64_t n = b->n_reads;
    TRY(compact_buffers(ctx, b));
    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    uint64_t h2d = 0;
    if (n) {
        TRY(reset_words(ctx));
        TRY(compact_copy_head(ctx, b, ctx->st, &h2d));
        TRY(compact_copy_range(ctx, b, 0, n, ctx->st, &h2d));
        TRY(compact_unpack_range(ctx, b, 0, n, ctx->st));
        if (ctx->batch_no_md) {                             /* K7 walks what K0 laid out: only once K0 has found it consistent */
            TRY(fetch_words(ctx)); TRY(device_error(ctx, "compact batch"));
            TRY(derive_md(ctx, 0));
        }
    }
    CU(cudaEventRecord(ctx->ev[1], ctx->st));
    if (n) { TRY(fetch_words(ctx)); TRY(device_error(ctx, "compact batch")); }
    else CU(cudaStreamSynchronize(ctx->st));
    ctx->have_batch = true;
    float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    ctx->stats.ms_h2d = ms; ctx->stats.h2d_bytes = h2d; ctx->stats.n_reads = n;
    return CBCG_OK;
}

extern "C" int cbcg_batch_upload(cbcg_ctx *ctx, const cbcg_batch *b) {
    if (!ctx) return CBCG_ERR_ARG;
    TRY(check_batch(ctx, b));
    if (b->n_reads && !b->md_off && !ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "a batch without MD needs the reference: cbcg_set_reference has not been called");
    CU(cudaSetDevice(ctx->device));
    const uint64_t n = b->n_reads;
    TRY(batch_prepare(ctx, b));
    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    uint64_t h2d = 0;
    TRY(batch_copy_range(ctx, b, 0, n, ctx->st, &h2d));
    const int scan_rc = batch_scan(ctx, b);               /* while the copies fly */
    const int md_rc = !scan_rc && n && ctx->batch_no_md ? derive_md(ctx, 0) : 0;   /* K7 on a checked batch; its time is part of ms_h2d */
    CU(cudaEventRecord(ctx->ev[1], ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    if (scan_rc) return scan_rc;                          /* nothing is left in flight that reads the caller's buffers */
    if (md_rc) return md_rc;
    ctx->have_batch = true;
    float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    ctx->stats.ms_h2d = ms; ctx->stats.h2d_bytes = h2d; ctx->stats.n_reads = n;
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ K1 */
static int reset_words(cbcg_ctx *ctx) {
    CU(cudaMemsetAsync(ctx->words.p, 0, sizeof(Words), ctx->st));
    return 0;
}
/* the device words -> their pinned host mirror, written by a kernel: a cudaMemcpyAsync would queue on the device -> host
   copy engine behind the decoded text of another batch in flight on this GPU (k2_coder.cu, "Small transfers by the SMs") */
static int fetch_words(cbcg_ctx *ctx) {
    static_assert(sizeof(Words) % 8 == 0 && sizeof(Words) / 8 <= 32, "Words travels as <= 32 64-bit words");
    if (launch_copy_words(ctx->hw, ctx->words.p, (uint32_t)(sizeof(Words) / 8), ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "word copy launch failed");
    CU(cudaStreamSynchronize(ctx->st));
    return 0;
}
/* pinned (cudaHostAlloc / cbcg_host_alloc / registered) host memory: the device reads and writes it in place */
static bool host_mapped(const void *p) {
    cudaPointerAttributes a;
    if (!p || cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost && a.devicePointer == p;
}

/* Runs K1 on the resident batch; on return ctx->hw->total_edits is valid. */
static int run_extract(cbcg_ctx *ctx) {
    const uint64_t n = ctx->db.n_reads;
    if (!ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "cbcg_set_reference has not been called");
    TRY(ensure(ctx, ctx->recs, (n + 1) * sizeof(cbcg_read_rec)));
    TRY(ensure(ctx, ctx->tile_desc, (extract_num_tiles(n) + 1) * 8));
    uint64_t cap = ctx->edits.cap / 2;
    const uint64_t guess = ctx->total_bases / 16 + 4096;          /* ~6 % of bases edited; grown on demand */
    if (cap < guess) { TRY(ensure(ctx, ctx->edits, guess * 2)); cap = ctx->edits.cap / 2; }
    for (int attempt = 0; attempt < 2; attempt++) {
        TRY(reset_words(ctx));
        if (launch_extract(ctx->db, ctx->dg, ctx->recs.as<cbcg_read_rec>(), ctx->edits.as<uint16_t>(), cap,
                           ctx->tile_desc.as<uint64_t>(), wptr<uint32_t>(ctx, W_OFF(ticket)), wptr<uint64_t>(ctx, W_OFF(total_edits)),
                           wptr<unsigned long long>(ctx, W_OFF(err)), ctx->st, ctx->kev[0], ctx->kev[1]))
            return fail(ctx, CBCG_ERR_CUDA, "K1 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        ctx->stats.kernel_launches++;
        TRY(fetch_words(ctx));
        cudaEventElapsedTime(&ctx->stats.ms_k1, ctx->kev[0], ctx->kev[1]);
        const unsigned long long v = ctx->hw->err;
        if (v && -(int)(v >> 40) == CBCG_ERR_CAPACITY && attempt == 0) {   /* edit array too small: the count is exact */
            TRY(ensure(ctx, ctx->edits, (ctx->hw->total_edits + 64) * 2));
            cap = ctx->edits.cap / 2;
            continue;
        }
        return device_error(ctx, "edit extraction");
    }
    return fail(ctx, CBCG_ERR_INTERNAL, "edit extraction: capacity retry failed");
}

/* K7 over the whole resident batch, one that came without MD: its MD pool and md_off. need: the pool's exact size when it
 * is known (the pipelined encode counted it), else 0. A pool too small for what K7 counts is grown to the exact size and
 * the batch derived once more, as run_extract does for edit entries. */
static int derive_md(cbcg_ctx *ctx, uint64_t need) {
    const uint64_t n = ctx->db.n_reads;
    TRY(ensure(ctx, ctx->tile_desc, (md_num_tiles(n) + 1) * 8));
    if (need + POOL_PAD > ctx->b_md.cap) TRY(ensure(ctx, ctx->b_md, need + POOL_PAD));
    for (int attempt = 0; attempt < 2; attempt++) {
        ctx->db.md = ctx->b_md.as<uint8_t>();
        TRY(reset_words(ctx));
        if (launch_md(ctx->db, ctx->dg, ctx->b_moff.as<uint64_t>(), ctx->b_md.as<uint8_t>(), ctx->b_md.cap - POOL_PAD, ctx->tile_desc.as<uint64_t>(),
                      wptr<uint32_t>(ctx, W_OFF(ticket)), wptr<uint64_t>(ctx, W_OFF(md_chain)), wptr<unsigned long long>(ctx, W_OFF(err)),
                      ctx->st, 0, n, nullptr))
            return fail(ctx, CBCG_ERR_CUDA, "K7 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        ctx->stats.kernel_launches++;
        TRY(fetch_words(ctx));
        const unsigned long long v = ctx->hw->err;
        if (v && -(int)(v >> 40) == CBCG_ERR_CAPACITY && attempt == 0) {   /* MD pool too small: the count is exact */
            TRY(ensure(ctx, ctx->b_md, ctx->hw->md_chain[0] + POOL_PAD));
            continue;
        }
        return device_error(ctx, "MD derivation");
    }
    return fail(ctx, CBCG_ERR_INTERNAL, "MD derivation: capacity retry failed");
}

extern "C" int cbcg_derive_md(cbcg_ctx *ctx, const cbcg_batch *batch, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!ctx || !batch || !out_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_derive_md: bad argument");
    *out_len = 0;
    cbcg_batch b = *batch;
    b.md_off = nullptr; b.md = nullptr;                   /* any MD the batch carries is ignored */
    TRY(cbcg_batch_upload(ctx, &b));
    const uint64_t n = ctx->db.n_reads;
    if (!n) return CBCG_OK;
    std::vector<uint64_t> off(n + 1);
    CU(cudaMemcpyAsync(off.data(), ctx->b_moff.p, (n + 1) * 8, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    *out_len = off[n] + n;
    if (!out || off[n] + n > out_cap) return fail(ctx, CBCG_ERR_CAPACITY, "derived MD is %llu bytes, room for %llu", (unsigned long long)(off[n] + n), (unsigned long long)out_cap);
    if (off[n]) CU(cudaMemcpyAsync(out, ctx->b_md.p, off[n], cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    for (uint64_t r = n; r-- > 0;) {                      /* in place, from the back: read r moves r bytes up, then its '\n' */
        memmove(out + off[r] + r, out + off[r], off[r + 1] - off[r]);
        out[off[r + 1] + r] = '\n';
    }
    return CBCG_OK;
}

extern "C" int cbcg_extract(cbcg_ctx *ctx, const cbcg_batch *batch, cbcg_read_rec *recs,
                            uint16_t *edits, uint64_t edits_cap, uint64_t *n_edits) {
    if (!ctx || !recs || (!edits && edits_cap) || !n_edits) return fail(ctx, CBCG_ERR_ARG, "cbcg_extract: bad argument");
    TRY(cbcg_batch_upload(ctx, batch));
    *n_edits = 0;
    if (!ctx->db.n_reads) return CBCG_OK;
    TRY(run_extract(ctx));
    const uint64_t ne = ctx->hw->total_edits;
    *n_edits = ne;
    if (ne > edits_cap) return fail(ctx, CBCG_ERR_CAPACITY, "cbcg_extract: %llu edit entries, room for %llu", (unsigned long long)ne, (unsigned long long)edits_cap);
    CU(cudaMemcpyAsync(recs, ctx->recs.p, ctx->db.n_reads * sizeof(cbcg_read_rec), cudaMemcpyDeviceToHost, ctx->st));
    if (ne) CU(cudaMemcpyAsync(edits, ctx->edits.p, ne * 2, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    ctx->stats.n_edits = ne;
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ blocks */
static void gens_from_blocks(cbcg_ctx *ctx, uint64_t nb) {
    ctx->gens.clear();
    ctx->max_block_reads = 0;
    for (uint64_t k = 0; k < nb; k++) {
        ctx->max_block_reads = std::max(ctx->max_block_reads, ctx->hblocks[k].n_reads);
        if (ctx->gens.empty() || ctx->hblocks[k].gen != ctx->hblocks[ctx->gens.back().first].gen) ctx->gens.push_back({ (uint32_t)k, 0u });
        ctx->gens.back().second++;
    }
}

/* Blocks of block_reads reads, never across a chromosome change. gen_mode 1: the first generations follow the
 * CBCG_GEN_* schedule (small blocks that bootstrap the model snapshots), the last one takes the rest. */
struct SizeStep { uint64_t r_limit; uint32_t block_reads; };    /* last-generation blocks that start below r_limit get this size */
static int cut_blocks(cbcg_ctx *ctx, uint32_t block_reads, uint32_t gen_mode, uint64_t *n_blocks_out,
                      const std::vector<SizeStep> *ramp = nullptr, bool upload = true) {
    const uint64_t n = ctx->db.n_reads;
    uint32_t sched_count[CBCG_GEN_MAX], sched_reads[CBCG_GEN_MAX], sched_last = 0;
    uint32_t split_gens = 0;
    const uint32_t n_sched = gen_mode ? cbcg_gen_schedule(n, ctx->layout, sched_count, sched_reads, &sched_last, &split_gens) : 0u;
    ctx->layout_mode = ctx->layout == 4u ? CBCG_MODE_SPLIT4 : (ctx->layout == 0u && gen_mode) ? CBCG_MODE_WITH_SPLIT_GENS(split_gens) : 0u;
    uint64_t bound = 1;
    uint32_t min_reads = block_reads;
    if (ramp) for (const SizeStep &st : *ramp) min_reads = std::min(min_reads, std::max(st.block_reads, 1u));
    if (block_reads) { for (const ChrRun &r : ctx->runs) bound += r.n / min_reads + 1; for (uint32_t g = 0; g < n_sched; g++) bound += sched_count[g]; }
    if (bound >= 0xffffffffull) return fail(ctx, CBCG_ERR_ARG, "too many blocks");
    TRY(ensure_hblocks(ctx, bound + 1));
    BlockDesc *hb = ctx->hblocks;
    uint64_t nb = 0;
    if (block_reads == 0) {
        memset(&hb[0], 0, sizeof(BlockDesc));
        hb[0].first_read = 0; hb[0].n_reads = (uint32_t)n; hb[0].chr = ctx->runs.empty() ? 0 : ctx->runs[0].chr;
        nb = 1;
    } else {
        uint32_t gen = 0, left = n_sched ? sched_count[0] : 0;
        size_t ramp_i = 0;
        for (const ChrRun &r : ctx->runs) {
            uint64_t o = 0;
            while (o < r.n) {
                uint32_t want = gen < n_sched ? sched_reads[gen] : block_reads;
                if (gen >= n_sched && ramp) {
                    while (ramp_i + 1 < ramp->size() && r.first + o >= (*ramp)[ramp_i].r_limit) ramp_i++;
                    want = (*ramp)[ramp_i].block_reads;
                }
                if (!want) want = 1;
                BlockDesc &d = hb[nb++];
                memset(&d, 0, sizeof d);
                d.first_read = (uint32_t)(r.first + o);
                d.n_reads = (uint32_t)std::min<uint64_t>(want, r.n - o);
                d.chr = r.chr; d.gen = gen;
                o += d.n_reads;
                if (gen < n_sched && --left == 0) { gen++; left = gen < n_sched ? sched_count[gen] : 0; }
            }
        }
    }
    gens_from_blocks(ctx, nb);
    TRY(ensure(ctx, ctx->blocks, (nb + 1) * sizeof(BlockDesc)));
    if (nb && upload) CU(cudaMemcpyAsync(ctx->blocks.p, hb, nb * sizeof(BlockDesc), cudaMemcpyHostToDevice, ctx->st));
    *n_blocks_out = nb;
    return 0;
}

/* CBCG_BLOCK_AUTO: reads per last-generation block such that the generation fills the GPU's resident block slots a
 * whole number of times. */
static uint32_t auto_block_reads(cbcg_ctx *ctx, uint64_t n, uint32_t gen_mode, uint64_t *slots_out = nullptr) {
    if (slots_out) *slots_out = 0;
    if (!gen_mode) return 1024u;
    uint32_t c[CBCG_GEN_MAX], r[CBCG_GEN_MAX], last = 0;
    const uint32_t k = cbcg_gen_schedule(n, ctx->layout, c, r, &last, nullptr);   /* what the <= 1 % budget leaves for the last generation */
    if (ctx->layout == 4u) return last;
    /* one warp per block: the last generation runs in whole waves of the GPU's resident warps (a few blocks beyond a wave
       cost a whole block time); rounded to fewer, larger blocks, never more */
    uint64_t early = 0;
    for (uint32_t g = 0; g < k; g++) early += (uint64_t)c[g] * r[g];
    const uint64_t rest = n > early ? n - early : 0;
    const uint64_t slots = coder_resident_blocks(ctx->device);
    if (slots_out) *slots_out = slots;
    if (!rest || !slots) return last;
    const uint64_t blocks = (rest + last - 1) / last;
    const uint64_t waves = std::max<uint64_t>(1, blocks / slots);
    if (blocks <= slots * waves) return last;
    return (uint32_t)std::min<uint64_t>((rest + waves * slots - 1) / (waves * slots), 16384u);
}
/* reads the early generations of the default cut hold (everything but the last generation) */
static uint64_t sched_early_reads(cbcg_ctx *ctx, uint64_t n, uint32_t *levels_out = nullptr) {
    uint32_t c[CBCG_GEN_MAX], r[CBCG_GEN_MAX], last = 0;
    const uint32_t k = cbcg_gen_schedule(n, ctx->layout, c, r, &last, nullptr);
    uint64_t early = 0;
    for (uint32_t g = 0; g < k; g++) early += (uint64_t)c[g] * r[g];
    if (levels_out) *levels_out = k;
    return early;
}
static int ensure_fin(cbcg_ctx *ctx, uint64_t nb) { return ensure(ctx, ctx->fin, (nb + 1) * fin_stride_bytes()); }
/* Interval buffer of the two-kernel encode (blocked containers): regions are addressed by absolute read and edit offsets
 * (k2_tri_off), so it is sized by the batch and the capacity of the edit array. */
static int ensure_tri(cbcg_ctx *ctx, CoderParams &p, uint64_t n, uint64_t nb) {
    TRY(ensure(ctx, ctx->tri, k2_tri_slots(n, ctx->edits.cap / 2, nb) * 16));
    p.tri = ctx->tri.as<K2Tri>();
    return 0;
}

/* Generations 0 .. last-1 of ctx->gens with the merges that build the snapshots; *snap_out = the snapshot the last
 * generation starts from. */
/* substreams of the blocks of the generation that block k belongs to */
static uint32_t gen_n_sub(const cbcg_ctx *ctx, uint32_t k) { return CBCG_BLOCK_NSUB(ctx->layout_mode, ctx->hblocks[k].gen); }

static int run_early_generations(cbcg_ctx *ctx, CoderParams p, uint8_t **snap_out, cudaStream_t st = nullptr) {
    if (!st) st = ctx->st;
    const uint64_t sb = snapshot_bytes(p.L);
    TRY(ensure(ctx, ctx->snap_a, sb)); TRY(ensure(ctx, ctx->snap_b, sb));
    uint8_t *cur = ctx->snap_a.as<uint8_t>(), *other = ctx->snap_b.as<uint8_t>();
    const uint32_t flag_target = cbcg_flag_target(ctx->max_block_reads);
    if (launch_snapshot_init(cur, p.L, st)) return fail(ctx, CBCG_ERR_CUDA, "snapshot init launch failed");
    ctx->stats.kernel_launches++;
    for (size_t g = 0; g + 1 < ctx->gens.size(); g++) {
        p.block_begin = ctx->gens[g].first; p.n_blocks = ctx->gens[g].second;
        p.n_sub = gen_n_sub(ctx, p.block_begin);
        p.snap = cur;
        if (launch_coder(p, st)) return fail(ctx, CBCG_ERR_CUDA, "K2 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        ctx->stats.kernel_launches += coder_launches(p);
        if (launch_merge(p.blocks, p.block_begin, p.n_blocks, p.L, cur, other, p.fin + (uint64_t)p.block_begin * fin_stride_bytes(), p.ws, p.err, flag_target, st))
            return fail(ctx, CBCG_ERR_CUDA, "merge launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        ctx->stats.kernel_launches += 4;
        std::swap(cur, other);
    }
    *snap_out = cur;
    return 0;
}

/* Runs the block coder (encode or decode) over all blocks of ctx->hblocks, generation by generation when primed:
 * blocks of generation g start from snapshot S_{g-1}; after each generation but the last the merge kernels build S_g. */
static int run_coder_generations(cbcg_ctx *ctx, CoderParams p, uint64_t nb, bool primed) {
    if (p.legacy || p.mode == 2u) {                          /* single-block stream / symbol lists: the warp kernel, no snapshot */
        p.block_begin = 0; p.n_blocks = (uint32_t)nb;
        if (launch_coder(p, ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "K2 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        ctx->stats.kernel_launches++;
        return 0;
    }
    /* blocked containers: every block starts from a snapshot. gen_mode 0: all of them from S_{-1}, the reference's initial
       state (one generation, run_early_generations only writes that snapshot). */
    (void)primed;
    if (ctx->gens.empty()) return 0;
    uint8_t *cur = nullptr;
    TRY(run_early_generations(ctx, p, &cur));
    p.block_begin = ctx->gens.back().first; p.n_blocks = ctx->gens.back().second;
    p.n_sub = gen_n_sub(ctx, p.block_begin);
    p.snap = cur; p.no_merge = 1u;                          /* the last generation: nobody merges its blocks */
    if (launch_coder(p, ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "K2 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    ctx->stats.kernel_launches += coder_launches(p);
    return 0;
}

static CoderParams coder_params(cbcg_ctx *ctx, uint32_t n_blocks, uint32_t L, int legacy, int mode) {
    CoderParams p;
    memset(&p, 0, sizeof p);
    p.n_blocks = n_blocks; p.L = L; p.legacy = legacy ? 1u : 0u; p.mode = (uint32_t)mode;
    p.blocks = ctx->blocks.as<BlockDesc>();
    p.recs = ctx->recs.as<cbcg_read_rec>();
    p.edits = ctx->edits.as<uint16_t>();
    p.genome = ctx->dg;
    p.ws = ctx->ws.as<uint8_t>();
    p.chr_names = ctx->g_names.as<uint8_t>();
    p.err = wptr<unsigned long long>(ctx, W_OFF(err));
    p.fin = ctx->fin.as<uint8_t>();                         /* callers ensure_fin(nb) before a blocked launch */
    p.layout_mode = legacy ? 0u : ctx->layout_mode;
    p.n_sub = 1u;                                           /* per launch: gen_n_sub() */
    p.indel_heavy = ctx->batch_indel_heavy ? 1u : 0u;
    return p;
}

/* opts->substreams: 1 = one stream per block, 4 = four substreams, 0 = the default: four in the narrow early generations of
 * a generation-primed container (they are latency-bound: three times faster as four short chains), one elsewhere */
static uint32_t opts_layout(const cbcg_encode_opts *o) { return o->substreams == CBCG_N_SUB ? 4u : (o->substreams == 0u && o->gen_mode == 1u) ? 0u : 1u; }
static int validate_opts(cbcg_ctx *ctx, const cbcg_encode_opts *o) {
    if (!o) return fail(ctx, CBCG_ERR_ARG, "NULL options");
    if (o->read_len_header == 0 || o->read_len_header > CBCG_MAX_READ_LEN) return fail(ctx, CBCG_ERR_ARG, "read_len_header must be in 1..%u", CBCG_MAX_READ_LEN);
    if (o->gen_mode > 1) return fail(ctx, CBCG_ERR_ARG, "gen_mode %u is not supported by this build", o->gen_mode);
    if (o->substreams != 0 && o->substreams != 1 && o->substreams != CBCG_N_SUB) return fail(ctx, CBCG_ERR_ARG, "substreams must be 0, 1 or %u", CBCG_N_SUB);
    return 0;
}

/* Container header + index of the blocks in ctx->hblocks (layout: DESIGN.md, "Container"), and the bookkeeping of
 * "the last encode" that cbcg_fetch_container / cbcg_decode_resident use. */
static void finish_encode(cbcg_ctx *ctx, const cbcg_encode_opts *opts, int legacy, bool fixed, uint64_t n, uint64_t n_edits,
                          uint64_t nb, uint64_t payload_total) {
    const uint32_t L = opts->read_len_header;
    cbcg_stats &S = ctx->stats;
    std::vector<uint8_t> &h = ctx->enc_head;
    h.clear();
    uint64_t n_syms = 0;
    for (uint64_t k = 0; k < nb; k++) n_syms += ctx->hblocks[k].n_symbols;
    if (!legacy) container_head(h, ctx->db.max_len, L, n, nb, ctx->names, opts->block_reads, opts->gen_mode | (fixed ? CBCG_MODE_FIXED_LEN : 0u) | ctx->layout_mode, ctx->hblocks);
    ctx->enc_L = L; ctx->enc_block_reads = opts->block_reads; ctx->enc_gen_mode = opts->gen_mode; ctx->enc_legacy = legacy;
    ctx->enc_max_len = ctx->db.max_len; ctx->enc_fixed = fixed ? 1u : 0u; ctx->enc_layout_mode = legacy ? 0u : ctx->layout_mode;
    ctx->enc_n_reads = n; ctx->enc_n_edits = n_edits; ctx->enc_n_blocks = nb; ctx->enc_payload_bytes = payload_total;
    ctx->have_encoded = true;
    S.n_reads = n; S.n_blocks = nb; S.n_edits = n_edits; S.n_symbols = n_syms;
    S.payload_bytes = payload_total; S.container_bytes = h.size() + payload_total;
}

/* ------------------------------------------------------------------------------------------------ encode */
/* Resident encode with the head of K1 split off (gen_mode 1, large batches): the early generations only need the
 * records of their own reads, so K1 runs on those first, and the rest of the batch is extracted on a side stream while
 * generations 0..3 (a few hundred CTAs at most) and their merges run on the main stream. Same cut, same container as the
 * one-stream order. The model workspace is sized from the head's edit density (one host round trip, as in the
 * pipelined host-buffer call); a batch whose tail is much dirtier than its head reports CBCG_ERR_CAPACITY / INTERNAL on
 * the device and the caller falls back to the one-stream order. CBCG_NO_OVERLAP=1 keeps the one-stream order. */
#define PIPE_FALLBACK 1            /* not an error: the caller takes the one-stream path */
static int pipe_init(cbcg_ctx *ctx);
static int encode_resident_overlapped(cbcg_ctx *ctx, const cbcg_encode_opts *opts) {
    const uint64_t n = ctx->db.n_reads;
    const uint32_t L = opts->read_len_header;
    const uint64_t tile = 128;                              /* K1 tile */
    uint32_t levels = 0;
    const uint64_t early = sched_early_reads(ctx, n, &levels);
    const uint64_t head_end = ((early + tile - 1) / tile + 1) * tile;   /* + one tile: the record after the last early block exists */
    if (n < 4 * head_end) return PIPE_FALLBACK;
    TRY(pipe_init(ctx));
    cbcg_stats &S = ctx->stats;
    uint64_t nb = 0;
    TRY(cut_blocks(ctx, opts->block_reads, 1, &nb));
    if (!levels || ctx->gens.size() != levels + 1u) return PIPE_FALLBACK;   /* chromosome runs too short for the schedule */
    const uint32_t last_first = ctx->gens.back().first, last_n = ctx->gens.back().second;
    if ((uint64_t)ctx->hblocks[last_first].first_read + tile > head_end) return PIPE_FALLBACK;
    const bool fixed = ctx->batch_min_len == L && ctx->db.max_len == L;
    TRY(ensure_fin(ctx, nb));

    const uint64_t edits_cap_guess = ctx->total_bases / 16 + 4096;
    TRY(ensure(ctx, ctx->recs, (n + 1) * sizeof(cbcg_read_rec)));
    TRY(ensure(ctx, ctx->tile_desc, ((n + tile - 1) / tile + 2) * 8));
    if (ctx->edits.cap / 2 < edits_cap_guess) TRY(ensure(ctx, ctx->edits, edits_cap_guess * 2));
    const uint64_t edits_cap = ctx->edits.cap / 2;
    TRY(ensure(ctx, ctx->out_off, (nb + 1) * 8));
    TRY(reset_words(ctx));
    uint64_t *chain = wptr<uint64_t>(ctx, W_OFF(chain));
    uint64_t *totals = wptr<uint64_t>(ctx, W_OFF(totals));
    uint32_t *ticket = wptr<uint32_t>(ctx, W_OFF(ticket));
    unsigned long long *err = wptr<unsigned long long>(ctx, W_OFF(err));
    cudaStream_t side = ctx->ps[1];

    /* K1 on the head; its edit total (chain[1]) gives the density the workspace is sized from */
    if (launch_extract(ctx->db, ctx->dg, ctx->recs.as<cbcg_read_rec>(), ctx->edits.as<uint16_t>(), edits_cap, ctx->tile_desc.as<uint64_t>(),
                       ticket, &chain[1], err, ctx->st, ctx->tev[0], ctx->tev[1], 0, head_end, nullptr))
        return fail(ctx, CBCG_ERR_CUDA, "K1 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    CU(cudaMemcpyAsync(&ctx->hw->total_edits, &chain[1], 8, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    const uint64_t proj = std::min<uint64_t>(edits_cap, (uint64_t)((double)ctx->hw->total_edits * ((double)n / (double)head_end) * 1.5) + 65536u);
    const uint64_t ws_cap = coder_ws_bytes_bound(L, n, proj, nb, 0, 1);
    const uint64_t pay_cap = coder_payload_bound(n, proj, nb, 0);
    TRY(ensure(ctx, ctx->ws, ws_cap)); TRY(ensure(ctx, ctx->scratch, pay_cap)); TRY(ensure(ctx, ctx->payload, pay_cap));
    CU(cudaEventRecord(ctx->ev[1], ctx->st));

    CoderParams p = coder_params(ctx, (uint32_t)nb, L, 0, 0);
    p.chr = const_cast<uint32_t *>(ctx->db.chr);
    p.payload = ctx->scratch.as<uint8_t>();
    p.lean = 1u; p.short_flush = 1u; p.primed = 1u; p.fixed_len = fixed ? 1u : 0u;
    TRY(ensure_tri(ctx, p, n, nb));
    /* high-priority stream: plan of the early blocks, generations 0..3. K1's grid fills every SM; without the priority
       the first generation's four CTAs queue behind all of it (measured: the overlap gained nothing). */
    cudaStream_t hp = ctx->hp;
    CU(cudaStreamWaitEvent(hp, ctx->ev[1], 0));
    CoderParams q = p;
    q.block_begin = 0; q.n_blocks = last_first;
    if (launch_plan(q, (uint32_t)head_end, 0, ws_cap, pay_cap, totals, hp, nullptr, &chain[1])) return fail(ctx, CBCG_ERR_CUDA, "plan launch failed");
    CU(cudaEventRecord(ctx->kev2[2], hp));
    CU(cudaEventRecord(ctx->ev[2], hp));
    /* side stream: K1 on the tail (everything before it on the main stream has completed: the synchronize above) */
    if (launch_extract(ctx->db, ctx->dg, ctx->recs.as<cbcg_read_rec>(), ctx->edits.as<uint16_t>(), edits_cap,
                       ctx->tile_desc.as<uint64_t>() + head_end / tile, ticket, &chain[0], err, side, ctx->kev[0], ctx->kev[1],
                       head_end, n, &chain[1]))
        return fail(ctx, CBCG_ERR_CUDA, "K1 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    uint8_t *snap = nullptr;
    TRY(run_early_generations(ctx, p, &snap, hp));
    CU(cudaEventRecord(ctx->dev2[2], hp));
    /* side stream: plan of the last generation, behind the tail's K1 and the early blocks' plan (its offsets carry on) */
    CU(cudaStreamWaitEvent(side, ctx->kev2[2], 0));
    q.block_begin = last_first; q.n_blocks = last_n;
    if (launch_plan(q, (uint32_t)n, 0, ws_cap, pay_cap, totals, side, totals, &chain[0])) return fail(ctx, CBCG_ERR_CUDA, "plan launch failed");
    CU(cudaEventRecord(ctx->dev2[1], side));
    CU(cudaStreamWaitEvent(ctx->st, ctx->dev2[1], 0));
    CU(cudaStreamWaitEvent(ctx->st, ctx->dev2[2], 0));
    q.snap = snap; q.n_sub = gen_n_sub(ctx, q.block_begin); q.no_merge = 1u;
    if (launch_coder(q, ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "K2 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    CU(cudaEventRecord(ctx->ev[3], ctx->st));
    if (launch_gather(p.blocks, (uint32_t)nb, ctx->scratch.as<uint8_t>(), ctx->payload.as<uint8_t>(), ctx->out_off.as<uint64_t>(), 1, ctx->layout_mode, ctx->st))
        return fail(ctx, CBCG_ERR_CUDA, "gather launch failed");
    S.kernel_launches += 6 + coder_launches(q);             /* K1 x 2, plan x 2, gather x 2, the last generation */
    CU(cudaEventRecord(ctx->ev[4], ctx->st));
    CU(cudaMemcpyAsync(ctx->hblocks, ctx->blocks.p, nb * sizeof(BlockDesc), cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(&ctx->hw->total_bytes, ctx->out_off.as<uint64_t>() + nb, 8, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(&ctx->hw->total_edits, &chain[0], 8, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaMemcpyAsync(&ctx->hw->err, err, 8, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    if (ctx->hw->err) {
        const int code = -(int)(ctx->hw->err >> 40);
        if (code == CBCG_ERR_CAPACITY || code == CBCG_ERR_INTERNAL) { S.retried = 1u; return PIPE_FALLBACK; }   /* projection too small */
        return device_error(ctx, "block coder");
    }
    float head_ms = 0, tail_ms = 0;
    cudaEventElapsedTime(&head_ms, ctx->tev[0], ctx->tev[1]);
    cudaEventElapsedTime(&tail_ms, ctx->kev[0], ctx->kev[1]);
    S.ms_k1 = head_ms + tail_ms;
    cudaEventElapsedTime(&S.ms_extract, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&S.ms_plan, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&S.ms_code, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&S.ms_gather, ctx->ev[3], ctx->ev[4]);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[4]);
    S.d2h_bytes += nb * sizeof(BlockDesc) + 24;
    finish_encode(ctx, opts, 0, fixed, n, ctx->hw->total_edits, nb, ctx->hw->total_bytes);
    return CBCG_OK;
}

extern "C" int cbcg_encode_resident(cbcg_ctx *ctx, const cbcg_encode_opts *opts) {
    if (!ctx) return CBCG_ERR_ARG;
    TRY(validate_opts(ctx, opts));
    if (!ctx->have_batch) return fail(ctx, CBCG_ERR_ARG, "no resident batch: call cbcg_batch_upload first");
    CU(cudaSetDevice(ctx->device));
    set_carveout_all(-1);
    const uint64_t n = ctx->db.n_reads;
    const int legacy = opts->block_reads == 0;
    const uint32_t L = opts->read_len_header;
    ctx->layout = legacy ? 1u : opts_layout(opts);
    cbcg_encode_opts auto_opts = *opts;
    if (opts->block_reads == CBCG_BLOCK_AUTO) {             /* last generation = a whole number of full waves */
        auto_opts.block_reads = auto_block_reads(ctx, n, opts->gen_mode);
        opts = &auto_opts;
    }
    ctx->have_encoded = false;
    cbcg_stats &S = ctx->stats;
    S.ms_extract = S.ms_plan = S.ms_code = S.ms_gather = S.ms_reconstruct = S.ms_d2h = S.ms_total = S.ms_k1 = S.ms_k3 = 0;
    S.kernel_launches = 0; S.d2h_bytes = 0; S.retried = 0;
    if (!ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "cbcg_set_reference has not been called");

    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    if (n && !legacy && opts->gen_mode == 1 && !getenv("CBCG_NO_OVERLAP")) {
        const int rc = encode_resident_overlapped(ctx, opts);
        if (rc != PIPE_FALLBACK) return rc;
        S.kernel_launches = 0; S.d2h_bytes = 0;
        if (ctx->pipe_ready) { CU(cudaStreamSynchronize(ctx->ps[1])); CU(cudaStreamSynchronize(ctx->hp)); }   /* nothing of the attempt is left in flight */
        CU(cudaEventRecord(ctx->ev[0], ctx->st));
    }
    uint64_t n_edits = 0, nb = 0;
    if (n) { TRY(run_extract(ctx)); n_edits = ctx->hw->total_edits; }
    CU(cudaEventRecord(ctx->ev[1], ctx->st));
    uint64_t payload_total = 0;
    bool fixed = false;
    if (n || legacy) {
        if (!n) {                                          /* legacy stream of an empty input: header + end marker */
            TRY(ensure(ctx, ctx->recs, sizeof(cbcg_read_rec))); TRY(ensure(ctx, ctx->edits, 64));
            CU(cudaMemsetAsync(ctx->recs.p, 0, sizeof(cbcg_read_rec), ctx->st));
            TRY(reset_words(ctx));
        }
        const bool primed = !legacy;                        /* blocked containers: every block starts from a snapshot (gen_mode 0: the initial one) */
        fixed = !legacy && ctx->batch_min_len == L && ctx->db.max_len == L;   /* CBCG_MODE_FIXED_LEN */
        TRY(cut_blocks(ctx, opts->block_reads, opts->gen_mode, &nb));
        if (!legacy) TRY(ensure_fin(ctx, nb));
        const uint64_t ws_cap = coder_ws_bytes_bound(L, n, n_edits, nb, legacy, primed);
        const uint64_t pay_cap = coder_payload_bound(n, n_edits, nb, legacy);
        TRY(ensure(ctx, ctx->ws, ws_cap));
        TRY(ensure(ctx, ctx->scratch, pay_cap));
        TRY(ensure(ctx, ctx->out_off, (nb + 1) * 8));
        CoderParams p = coder_params(ctx, (uint32_t)nb, L, legacy, 0);
        p.chr = const_cast<uint32_t *>(ctx->db.chr);
        p.payload = ctx->scratch.as<uint8_t>();
        p.lean = legacy ? 0u : 1u; p.short_flush = legacy ? 0u : 1u; p.primed = primed ? 1u : 0u; p.fixed_len = fixed ? 1u : 0u;
        if (!legacy) TRY(ensure_tri(ctx, p, n, nb));
        if (launch_plan(p, (uint32_t)n, n_edits, ws_cap, pay_cap, wptr<uint64_t>(ctx, W_OFF(totals)), ctx->st))
            return fail(ctx, CBCG_ERR_CUDA, "plan launch failed");
        CU(cudaEventRecord(ctx->ev[2], ctx->st));
        TRY(run_coder_generations(ctx, p, nb, primed));
        CU(cudaEventRecord(ctx->ev[3], ctx->st));
        /* compact payload: bounded by the scratch size */
        TRY(ensure(ctx, ctx->payload, pay_cap));
        if (launch_gather(p.blocks, (uint32_t)nb, ctx->scratch.as<uint8_t>(), ctx->payload.as<uint8_t>(), ctx->out_off.as<uint64_t>(), legacy ? 0 : 1, ctx->layout_mode, ctx->st))
            return fail(ctx, CBCG_ERR_CUDA, "gather launch failed");
        S.kernel_launches += 3;
        CU(cudaEventRecord(ctx->ev[4], ctx->st));
        CU(cudaMemcpyAsync(ctx->hblocks, ctx->blocks.p, nb * sizeof(BlockDesc), cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaMemcpyAsync(&ctx->hw->total_bytes, ctx->out_off.as<uint64_t>() + nb, 8, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaMemcpyAsync(&ctx->hw->err, wptr<unsigned long long>(ctx, W_OFF(err)), 8, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
        TRY(device_error(ctx, "block coder"));
        payload_total = ctx->hw->total_bytes;
        S.d2h_bytes += nb * sizeof(BlockDesc) + 16;
    } else {
        CU(cudaEventRecord(ctx->ev[2], ctx->st)); CU(cudaEventRecord(ctx->ev[3], ctx->st)); CU(cudaEventRecord(ctx->ev[4], ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
    }
    cudaEventElapsedTime(&S.ms_extract, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&S.ms_plan, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&S.ms_code, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&S.ms_gather, ctx->ev[3], ctx->ev[4]);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[4]);

    finish_encode(ctx, opts, legacy, fixed, n, n_edits, nb, payload_total);
    return CBCG_OK;
}

extern "C" int cbcg_fetch_container(cbcg_ctx *ctx, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!ctx || !out_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_fetch_container: bad argument");
    if (!ctx->have_encoded) return fail(ctx, CBCG_ERR_ARG, "nothing encoded yet");
    const uint64_t total = ctx->enc_head.size() + ctx->enc_payload_bytes;
    *out_len = total;
    if (total > out_cap || (!out && total)) return fail(ctx, CBCG_ERR_CAPACITY, "container is %llu bytes, room for %llu", (unsigned long long)total, (unsigned long long)out_cap);
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventRecord(ctx->ev[5], ctx->st));
    if (ctx->enc_payload_bytes) {
        if (host_mapped(out)) {                              /* pinned buffer: written in place by the SMs, no copy-engine queue */
            if (launch_d2h_bytes(out + ctx->enc_head.size(), ctx->payload.p, ctx->enc_payload_bytes, ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "container copy launch failed");
        } else CU(cudaMemcpyAsync(out + ctx->enc_head.size(), ctx->payload.p, ctx->enc_payload_bytes, cudaMemcpyDeviceToHost, ctx->st));
    }
    if (!ctx->enc_head.empty()) memcpy(out, ctx->enc_head.data(), ctx->enc_head.size());
    CU(cudaEventRecord(ctx->ev[6], ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    cudaEventElapsedTime(&ctx->stats.ms_d2h, ctx->ev[5], ctx->ev[6]);
    ctx->stats.d2h_bytes += ctx->enc_payload_bytes;
    return CBCG_OK;
}

/* Header + per-block index of the last encode (no payload): what a shard contributes to the container index. */
extern "C" int cbcg_fetch_index(cbcg_ctx *ctx, uint8_t *out, uint64_t out_cap, uint64_t *out_len, uint64_t *payload_bytes) {
    if (!ctx || !out_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_fetch_index: bad argument");
    if (!ctx->have_encoded) return fail(ctx, CBCG_ERR_ARG, "nothing encoded yet");
    *out_len = ctx->enc_head.size();
    if (payload_bytes) *payload_bytes = ctx->enc_payload_bytes;
    if (ctx->enc_head.size() > out_cap || (!out && !ctx->enc_head.empty())) return fail(ctx, CBCG_ERR_CAPACITY, "index is %zu bytes", ctx->enc_head.size());
    if (!ctx->enc_head.empty()) memcpy(out, ctx->enc_head.data(), ctx->enc_head.size());
    return CBCG_OK;
}

extern "C" uint64_t cbcg_encode_bound(const cbcg_batch *b, const cbcg_encode_opts *o) {
    if (!b || !o) return 0;
    /* Practical bound: one byte per base plus 16 per read is four times the 2-bit packing of the
       reads. A larger output makes cbcg_encode return CBCG_ERR_CAPACITY with the exact size in *out_len;
       cbcg_fetch_container then retrieves it without re-encoding. */
    const uint64_t n = b->n_reads;
    const uint64_t bases = n ? b->seq_off[n] - b->seq_off[0] : 0;
    const uint64_t nb = o->block_reads ? (n / o->block_reads + MAX_CHR + 2) : 1;
    return 4096 + (uint64_t)MAX_CHR * 16 + nb * 32 + n * 16 + bases;
}

/* ------------------------------------------------------------------------------------------------ pipelined encode
 * cbcg_encode on a large batch with automatic block size: the batch crosses PCIe in chunks of whole K1 tiles on a copy
 * stream; K1 and the block plan follow chunk by chunk, the early generations are coded while the rest of the batch is
 * still on the link, and the last generation is launched group by group (one side stream each) as its reads arrive.
 * Last-generation blocks shrink towards the end of the batch (the ramp), so that the blocks whose reads arrive last are
 * the ones that take least time: all groups end together shortly after the last byte has landed. The same layout lets
 * cbcg_decode start returning text while the large blocks are still being decoded. The cut is recorded in the
 * container's index like any other; the coded bits of a block depend only on its reads and its generation. */
#define PIPE_CHUNKS 5u             /* tail chunks (after the head that feeds the early generations); <= PIPE_MAX - 1 */
/* shares of the tail per chunk. Shrinking shares (0.30 .. 0.10) with a steeper ramp were measured and did not pay: a
 * group ends with its slowest block, and small blocks spread more (15.2 + 16.1 ms against 15.6 + 15.7 ms for equal shares). */
static const double PIPE_SHARE[PIPE_CHUNKS] = { 0.20, 0.20, 0.20, 0.20, 0.20 };
static uint64_t pipe_min_reads() {
    const char *e = getenv("CBCG_PIPE_MIN_READS");
    return e ? strtoull(e, nullptr, 10) : (1ull << 20);
}
/* Last-generation block size per tail chunk, as multiples of the mean (normalised below so that all blocks stay
 * co-resident). Convex: the last two chunks' blocks are much the shortest, so that the encoder is done soon after the
 * last byte has landed and the decoder has its first text early enough to keep the link busy to the end. Measured on
 * config 2 (encode + decode, ms): linear 1.3 .. 0.7: 14.09 + 14.53; this: 13.97 + 13.68; {1.3,1.2,1.0,0.7,0.45}: 14.24 + 13.51;
 * {1.4,1.25,1.0,0.7,0.45}: 14.18 + 13.53; {1.35,1.25,1.0,0.65,0.4}: 14.22 + 13.72; {1.3,1.25,1.1,0.7,0.4}: 14.42 + 14.75. */
static const double PIPE_MULT[PIPE_CHUNKS] = { 1.3, 1.2, 1.0, 0.6, 0.45 };
/* a compact batch is on the device after a third of the time: the encoder no longer waits for the link, a flatter ramp
   (which the decoder still wants: small blocks decode first and their text goes out while the large ones run) */
static const double PIPE_MULT_COMPACT[PIPE_CHUNKS] = { 1.15, 1.1, 1.0, 0.8, 0.6 };
static int pipe_init(cbcg_ctx *ctx) {
    if (ctx->pipe_ready) return 0;
    CU(cudaStreamCreateWithFlags(&ctx->cs, cudaStreamNonBlocking));
    for (auto &s : ctx->ps) CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    { int lo = 0, hi = 0; CU(cudaDeviceGetStreamPriorityRange(&lo, &hi)); CU(cudaStreamCreateWithPriority(&ctx->hp, cudaStreamNonBlocking, hi)); }
    for (auto &e : ctx->cev) CU(cudaEventCreate(&e));
    for (auto &e : ctx->kev2) CU(cudaEventCreate(&e));
    for (auto &e : ctx->dev2) CU(cudaEventCreate(&e));
    for (auto &e : ctx->tev) CU(cudaEventCreate(&e));
    ctx->pipe_ready = true;
    return 0;
}
/* Error exit of a pipelined call: nothing that touches the caller's buffers (or races the next call) stays in flight. */
static void pipe_drain(cbcg_ctx *ctx) {
    if (ctx->pipe_ready) {
        cudaStreamSynchronize(ctx->cs); cudaStreamSynchronize(ctx->hp);
        for (auto &s : ctx->ps) cudaStreamSynchronize(s);
    }
    cudaStreamSynchronize(ctx->st);
    (void)cudaGetLastError();
}
static int encode_pipelined(cbcg_ctx *ctx, const BatchSrc &src, const cbcg_encode_opts *opts) {
    const uint64_t n = src.n;
    ctx->layout = opts_layout(opts);
    const uint32_t L = opts->read_len_header;
    const uint64_t tile = 128;                              /* K1 tile: chunk boundaries are whole tiles */
    uint32_t levels = 0;
    const uint64_t early = sched_early_reads(ctx, n, &levels);
    if (n < early + tile * (PIPE_CHUNKS + 1)) return PIPE_FALLBACK;
    if (!ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "cbcg_set_reference has not been called");   /* before any copy is queued */
    TRY(pipe_init(ctx));
    TRY(src_prepare(ctx, src));
    set_carveout_all(100);
    cbcg_stats &S = ctx->stats;

    /* chunks: [0] = the head (early generations + one tile, so that the record after the last early block exists),
       [1..PIPE_CHUNKS] = the tail in equal parts */
    uint64_t cut[PIPE_CHUNKS + 2];
    const uint64_t head_end = ((early + tile - 1) / tile + 1) * tile;
    cut[0] = 0; cut[1] = head_end;
    /* tail chunks by their share of the tail (PIPE_SHARE) */
    {
        double acc = 0;
        for (uint32_t c = 1; c <= PIPE_CHUNKS; c++) {
            acc += PIPE_SHARE[c - 1];
            cut[c + 1] = c == PIPE_CHUNKS ? n : head_end + (uint64_t)((double)(n - head_end) * acc) / tile * tile;
        }
    }
    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    CU(cudaStreamWaitEvent(ctx->cs, ctx->ev[0], 0));        /* copies start after whatever the caller left on the main stream */
    uint64_t h2d = 0;
    if (src.compact) TRY(compact_copy_head(ctx, src.compact, ctx->cs, &h2d));
    for (uint32_t c = 0; c <= PIPE_CHUNKS; c++) {
        TRY(src_copy_range(ctx, src, cut[c], cut[c + 1], ctx->cs, &h2d));
        CU(cudaEventRecord(ctx->cev[c], ctx->cs));
    }
    if (src.full) TRY(batch_scan(ctx, src.full));           /* while the copies fly (a compact batch brings its figures with it) */
    const bool fixed = ctx->batch_min_len == L && ctx->db.max_len == L;

    /* the cut: early generations on their schedule, then the ramp */
    uint64_t slots = 0;
    cbcg_encode_opts used = *opts;
    used.block_reads = auto_block_reads(ctx, n, 1, &slots);
    std::vector<SizeStep> ramp;
    const double *mult = src.compact ? PIPE_MULT_COMPACT : PIPE_MULT;
    double inv = 0;
    for (uint32_t c = 0; c < PIPE_CHUNKS; c++) inv += PIPE_SHARE[c] / mult[c];
    /* inv > 1: more blocks than resident slots, the last ones would queue */
    for (uint32_t c = 1; c <= PIPE_CHUNKS; c++) {
        const double m = mult[c - 1] * (inv > 1.0 ? inv : 1.0);
        ramp.push_back({ cut[c + 1], (uint32_t)std::max(64.0, std::min(16384.0, m * used.block_reads)) });
    }
    uint64_t nb = 0;
    TRY(cut_blocks(ctx, used.block_reads, 1, &nb, &ramp, false));
    if (!levels || ctx->gens.size() != levels + 1u) return PIPE_FALLBACK;   /* chromosome runs too short for the schedule */
    TRY(ensure_fin(ctx, nb));
    const BlockDesc *hb = ctx->hblocks;
    const uint32_t last_first = ctx->gens.back().first, last_n = ctx->gens.back().second;
    if ((uint64_t)hb[last_first].first_read + tile > head_end) return PIPE_FALLBACK;
    /* groups of last-generation blocks: group c = the blocks that end inside chunk c + 1 or before (not yet taken) */
    uint32_t gb[PIPE_CHUNKS + 1]; gb[0] = last_first;
    {
        uint32_t k = last_first;
        for (uint32_t c = 1; c <= PIPE_CHUNKS; c++) {
            while (k < last_first + last_n && (uint64_t)hb[k].first_read + hb[k].n_reads <= cut[c + 1]) k++;
            /* whole CTAs (4 blocks) per group, so that the groups together need no more CTAs than one launch would:
               a CTA beyond the resident slots starts when the first block anywhere retires and ends a block late */
            if (c < PIPE_CHUNKS) k = last_first + ((k - last_first) & ~3u);
            gb[c] = k;
        }
        if (gb[PIPE_CHUNKS] != last_first + last_n) return fail(ctx, CBCG_ERR_INTERNAL, "pipelined encode: block groups do not cover the cut");
    }

    /* buffers (sized from bounds: no host round trip between the stages) */
    const uint64_t edits_cap_guess = ctx->total_bases / 16 + 4096;
    TRY(ensure(ctx, ctx->recs, (n + 1) * sizeof(cbcg_read_rec)));
    TRY(ensure(ctx, ctx->tile_desc, ((n + tile - 1) / tile + 1) * 8));
    if (ctx->edits.cap / 2 < edits_cap_guess) TRY(ensure(ctx, ctx->edits, edits_cap_guess * 2));
    const uint64_t edits_cap = ctx->edits.cap / 2;
    uint64_t ws_cap = 0, pay_cap = 0;                       /* sized once the head chunk has told the edit density */
    TRY(ensure(ctx, ctx->out_off, (nb + 1) * 8));
    TRY(ensure(ctx, ctx->blocks, (nb + 1) * sizeof(BlockDesc)));
    S.ms_extract = S.ms_plan = S.ms_code = S.ms_gather = S.ms_reconstruct = S.ms_d2h = S.ms_total = S.ms_k1 = S.ms_k3 = 0;
    S.kernel_launches = 0; S.d2h_bytes = 0;

    TRY(reset_words(ctx));
    /* the descriptors are read from pinned host memory by a kernel: a cudaMemcpyAsync would queue on the host -> device
       copy engine behind every chunk enqueued above */
    if (launch_copy16(ctx->blocks.p, hb, nb * sizeof(BlockDesc), ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "descriptor copy launch failed");
    CoderParams p = coder_params(ctx, (uint32_t)nb, L, 0, 0);
    p.chr = const_cast<uint32_t *>(ctx->db.chr);
    p.payload = ctx->scratch.as<uint8_t>();
    p.lean = 1u; p.short_flush = 1u; p.primed = 1u; p.fixed_len = fixed ? 1u : 0u;
    uint64_t *chain = wptr<uint64_t>(ctx, W_OFF(chain));
    uint64_t *totals = wptr<uint64_t>(ctx, W_OFF(totals));
    uint8_t *snap = nullptr;
    uint64_t tile_off = 0;
    for (uint32_t c = 0; c <= PIPE_CHUNKS; c++) {
        CU(cudaStreamWaitEvent(ctx->st, ctx->cev[c], 0));
        if (src.compact) TRY(compact_unpack_range(ctx, src.compact, cut[c], cut[c + 1], ctx->st));   /* 2-bit SEQ, lengths, runs -> the SoA batch */
        if (ctx->batch_no_md) {                              /* K7: the chunk's MD, continuing the previous chunk's */
            uint64_t *mdc = wptr<uint64_t>(ctx, W_OFF(md_chain));
            if (launch_md(ctx->db, ctx->dg, ctx->b_moff.as<uint64_t>(), ctx->b_md.as<uint8_t>(), ctx->b_md.cap - POOL_PAD,
                          ctx->tile_desc.as<uint64_t>() + tile_off, wptr<uint32_t>(ctx, W_OFF(ticket)), &mdc[(c + 1u) & 1u],
                          wptr<unsigned long long>(ctx, W_OFF(err)), ctx->st, cut[c], cut[c + 1], c ? &mdc[c & 1u] : nullptr))
                return fail(ctx, CBCG_ERR_CUDA, "K7 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
            S.kernel_launches++;
        }
        /* K1 on the chunk; its edit entries continue the previous chunk's */
        if (launch_extract(ctx->db, ctx->dg, ctx->recs.as<cbcg_read_rec>(), ctx->edits.as<uint16_t>(), edits_cap,
                           ctx->tile_desc.as<uint64_t>() + tile_off, wptr<uint32_t>(ctx, W_OFF(ticket)), &chain[(c + 1u) & 1u],
                           wptr<unsigned long long>(ctx, W_OFF(err)), ctx->st, nullptr, nullptr, cut[c], cut[c + 1],
                           c ? &chain[c & 1u] : nullptr))
            return fail(ctx, CBCG_ERR_CUDA, "K1 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        tile_off += (cut[c + 1] - cut[c] + tile - 1) / tile;
        S.kernel_launches++;
        if (c == 0) {
            /* the model workspace is bounded by the number of edit entries: project it from the head's (the one host
               round trip of the pipeline; the copies go on meanwhile). Too small a projection shows up as a device
               error and the call falls back to the one-stream path. */
            CU(cudaMemcpyAsync(&ctx->hw->total_edits, &chain[1], 8, cudaMemcpyDeviceToHost, ctx->st));
            CU(cudaStreamSynchronize(ctx->st));
            const uint64_t proj = std::min<uint64_t>(edits_cap, (uint64_t)((double)ctx->hw->total_edits * ((double)n / (double)head_end) * 1.5) + 65536u);
            ws_cap = coder_ws_bytes_bound(L, n, proj, nb, 0, 1);
            pay_cap = coder_payload_bound(n, proj, nb, 0);
            TRY(ensure(ctx, ctx->ws, ws_cap)); TRY(ensure(ctx, ctx->scratch, pay_cap)); TRY(ensure(ctx, ctx->payload, pay_cap));
            p.ws = ctx->ws.as<uint8_t>(); p.payload = ctx->scratch.as<uint8_t>();
            TRY(ensure_tri(ctx, p, n, nb));
        }
        /* plan of the blocks that are now complete */
        CoderParams q = p;
        q.block_begin = c ? gb[c - 1] : 0u; q.n_blocks = c ? gb[c] - gb[c - 1] : last_first;
        if (q.n_blocks) {
            if (launch_plan(q, (uint32_t)cut[c + 1], 0, ws_cap, pay_cap, totals, ctx->st, c ? totals : nullptr, &chain[(c + 1u) & 1u]))
                return fail(ctx, CBCG_ERR_CUDA, "plan launch failed");
            S.kernel_launches++;
        }
        if (c == 0) {                                        /* generations 0 .. 3 while the tail is on the link */
            TRY(run_early_generations(ctx, p, &snap));
        } else if (q.n_blocks) {
            CU(cudaEventRecord(ctx->kev2[c], ctx->st));
            cudaStream_t sd = ctx->ps[c % PIPE_MAX];
            CU(cudaStreamWaitEvent(sd, ctx->kev2[c], 0));
            q.snap = snap; q.n_sub = gen_n_sub(ctx, q.block_begin); q.no_merge = 1u;
            if (launch_coder(q, sd)) return fail(ctx, CBCG_ERR_CUDA, "K2 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
            S.kernel_launches += coder_launches(q);
            CU(cudaEventRecord(ctx->dev2[c], sd));
        }
    }
    for (uint32_t c = 1; c <= PIPE_CHUNKS; c++) if (gb[c] > gb[c - 1]) CU(cudaStreamWaitEvent(ctx->st, ctx->dev2[c], 0));
    if (launch_gather(p.blocks, (uint32_t)nb, ctx->scratch.as<uint8_t>(), ctx->payload.as<uint8_t>(), ctx->out_off.as<uint64_t>(), 1, ctx->layout_mode, ctx->st))
        return fail(ctx, CBCG_ERR_CUDA, "gather launch failed");
    S.kernel_launches += 2;
    CU(cudaEventRecord(ctx->ev[4], ctx->st));
    /* results to the pinned host mirrors by kernels, not by the device -> host copy engine (another batch's text may be
       queued there: k2_coder.cu, "Small transfers by the SMs") */
    if (launch_copy16(ctx->hblocks, ctx->blocks.p, nb * sizeof(BlockDesc), ctx->st) ||
        launch_copy_words(&ctx->hw->total_bytes, ctx->out_off.as<uint64_t>() + nb, 1, ctx->st) ||
        launch_copy_words(&ctx->hw->total_edits, &chain[(PIPE_CHUNKS + 1u) & 1u], 1, ctx->st) ||
        launch_copy_words(&ctx->hw->err, wptr<unsigned long long>(ctx, W_OFF(err)), 1, ctx->st) ||
        (ctx->batch_no_md && launch_copy_words(&ctx->hw->md_chain[0], wptr<uint64_t>(ctx, W_OFF(md_chain)) + ((PIPE_CHUNKS + 1u) & 1u), 1, ctx->st)))
        return fail(ctx, CBCG_ERR_CUDA, "result copy launch failed");
    CU(cudaStreamSynchronize(ctx->st));
    ctx->have_batch = true;
    if (getenv("CBCG_PIPE_TRACE")) {                        /* when each chunk landed, was extracted and planned, and was coded */
        for (uint32_t c = 0; c <= PIPE_CHUNKS; c++) {
            float a = 0, k = 0, d = 0;
            cudaEventElapsedTime(&a, ctx->ev[0], ctx->cev[c]);
            if (c && gb[c] > gb[c - 1]) { cudaEventElapsedTime(&k, ctx->ev[0], ctx->kev2[c]); cudaEventElapsedTime(&d, ctx->ev[0], ctx->dev2[c]); }
            fprintf(stderr, "[cbcg pipe enc] chunk %u reads %llu..%llu blocks %u size %u: copied %.2f ms, planned %.2f ms, coded %.2f ms\n", c,
                    (unsigned long long)cut[c], (unsigned long long)cut[c + 1], c ? gb[c] - gb[c - 1] : last_first,
                    c ? ramp[c - 1].block_reads : 0u, a, k, d);
        }
        float t = 0; cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[4]); fprintf(stderr, "[cbcg pipe enc] gathered %.2f ms\n", t);
    }
    S.h2d_bytes = h2d; S.d2h_bytes = nb * sizeof(BlockDesc) + 24;
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[4]);
    if (ctx->hw->err) {
        const int code = -(int)(ctx->hw->err >> 40);
        /* edit array or workspace guessed too small: the batch is resident now, take the one-stream path */
        if (code == CBCG_ERR_CAPACITY || code == CBCG_ERR_INTERNAL) return PIPE_FALLBACK;
        return device_error(ctx, "pipelined encode");
    }
    finish_encode(ctx, &used, 0, fixed, n, ctx->hw->total_edits, nb, ctx->hw->total_bytes);
    return CBCG_OK;
}

static int encode_from(cbcg_ctx *ctx, const BatchSrc &src, const cbcg_encode_opts *opts, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!ctx || !out_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_encode: bad argument");
    TRY(validate_opts(ctx, opts));
    if (src.compact) TRY(check_compact(ctx, src.compact)); else TRY(check_batch(ctx, src.full));
    if (opts->block_reads == CBCG_BLOCK_AUTO && opts->gen_mode == 1 && src.n >= pipe_min_reads()) {
        CU(cudaSetDevice(ctx->device));
        const int rc = encode_pipelined(ctx, src, opts);
        if (rc < 0) { pipe_drain(ctx); return rc; }          /* copies from the caller's batch may still be queued */
        if (rc == CBCG_OK) return cbcg_fetch_container(ctx, out, out_cap, out_len);
        if (ctx->have_batch) {                              /* fallback with the batch already resident */
            /* without MD: a pool that overflowed holds empty MD for the reads past its end; derive it whole at the size counted */
            if (ctx->batch_no_md) TRY(derive_md(ctx, ctx->hw->md_chain[0]));
            TRY(cbcg_encode_resident(ctx, opts));
            return cbcg_fetch_container(ctx, out, out_cap, out_len);
        }
    }
    if (src.compact) TRY(cbcg_batch_upload_compact(ctx, src.compact)); else TRY(cbcg_batch_upload(ctx, src.full));
    const float ms_h2d = ctx->stats.ms_h2d; const uint64_t h2d = ctx->stats.h2d_bytes;
    TRY(cbcg_encode_resident(ctx, opts));
    ctx->stats.ms_h2d = ms_h2d; ctx->stats.h2d_bytes = h2d;
    return cbcg_fetch_container(ctx, out, out_cap, out_len);
}
extern "C" int cbcg_encode(cbcg_ctx *ctx, const cbcg_batch *batch, const cbcg_encode_opts *opts,
                           uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!batch) return fail(ctx, CBCG_ERR_ARG, "NULL batch");
    const BatchSrc src = { batch, nullptr, batch->n_reads };
    return encode_from(ctx, src, opts, out, out_cap, out_len);
}
extern "C" int cbcg_encode_compact(cbcg_ctx *ctx, const cbcg_batch_compact *batch, const cbcg_encode_opts *opts,
                                   uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!batch) return fail(ctx, CBCG_ERR_ARG, "NULL batch");
    const BatchSrc src = { nullptr, batch, batch->n_reads };
    return encode_from(ctx, src, opts, out, out_cap, out_len);
}

/* ------------------------------------------------------------------------------------------------ symbol lists */
extern "C" int cbcg_extract_symbols(cbcg_ctx *ctx, const cbcg_batch *batch, const cbcg_encode_opts *opts,
                                    cbcg_symbol *symbols, uint64_t symbols_cap, uint64_t *n_symbols,
                                    uint64_t *block_sym_count, uint64_t blocks_cap, uint64_t *n_blocks) {
    if (!ctx || !n_symbols || (!symbols && symbols_cap)) return fail(ctx, CBCG_ERR_ARG, "cbcg_extract_symbols: bad argument");
    TRY(validate_opts(ctx, opts));
    TRY(cbcg_batch_upload(ctx, batch));
    const uint64_t n = ctx->db.n_reads;
    const int legacy = opts->block_reads == 0;
    ctx->layout = legacy ? 1u : opts_layout(opts);
    *n_symbols = 0; if (n_blocks) *n_blocks = 0;
    uint64_t n_edits = 0, nb = 0;
    if (n) { TRY(run_extract(ctx)); n_edits = ctx->hw->total_edits; }
    else if (!legacy) return CBCG_OK;
    else {
        TRY(ensure(ctx, ctx->recs, sizeof(cbcg_read_rec))); TRY(ensure(ctx, ctx->edits, 64));
        CU(cudaMemsetAsync(ctx->recs.p, 0, sizeof(cbcg_read_rec), ctx->st));
        TRY(reset_words(ctx));
    }
    TRY(cut_blocks(ctx, opts->block_reads, opts->gen_mode, &nb));
    const uint64_t list_cap = 12u * n + 2u * n_edits + nb * 8u + (legacy ? 136u + 2048u : 0u) + 64u;
    TRY(ensure(ctx, ctx->symbols, list_cap * sizeof(cbcg_symbol)));
    TRY(ensure(ctx, ctx->ws, 4096));
    CoderParams p = coder_params(ctx, (uint32_t)nb, opts->read_len_header, legacy, 2);
    p.chr = const_cast<uint32_t *>(ctx->db.chr);
    p.symbols = ctx->symbols.as<cbcg_symbol>();
    if (launch_plan(p, (uint32_t)n, n_edits, ~0ull, ~0ull, wptr<uint64_t>(ctx, W_OFF(totals)), ctx->st))
        return fail(ctx, CBCG_ERR_CUDA, "plan launch failed");
    if (launch_coder(p, ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "K2 (list) launch failed");
    CU(cudaMemcpyAsync(ctx->hblocks, ctx->blocks.p, nb * sizeof(BlockDesc), cudaMemcpyDeviceToHost, ctx->st));
    TRY(fetch_words(ctx));
    TRY(device_error(ctx, "symbol emission"));
    if (ctx->hw->totals[2] > list_cap) return fail(ctx, CBCG_ERR_INTERNAL, "symbol list bound exceeded");
    uint64_t total = 0;
    for (uint64_t k = 0; k < nb; k++) total += ctx->hblocks[k].n_symbols;
    *n_symbols = total;
    if (n_blocks) *n_blocks = nb;
    if (total > symbols_cap) return fail(ctx, CBCG_ERR_CAPACITY, "%llu symbols, room for %llu", (unsigned long long)total, (unsigned long long)symbols_cap);
    if (block_sym_count && nb > blocks_cap) return fail(ctx, CBCG_ERR_CAPACITY, "%llu blocks, room for %llu", (unsigned long long)nb, (unsigned long long)blocks_cap);
    uint64_t o = 0;
    for (uint64_t k = 0; k < nb; k++) {
        const BlockDesc &b = ctx->hblocks[k];
        if (b.n_symbols)
            CU(cudaMemcpyAsync(symbols + o, ctx->symbols.as<cbcg_symbol>() + b.sym_off, (size_t)b.n_symbols * sizeof(cbcg_symbol), cudaMemcpyDeviceToHost, ctx->st));
        if (block_sym_count) block_sym_count[k] = b.n_symbols;
        o += b.n_symbols;
    }
    CU(cudaStreamSynchronize(ctx->st));
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ decode */
struct Container {
    uint32_t max_len, L, n_blocks, n_chr, block_reads, gen_mode, fixed_len, layout_mode;
    uint64_t n_reads;
    uint64_t index_off, index_bytes, payload_off;
    std::vector<uint32_t> chr_map;             /* container ordinal -> genome ordinal */
};

/* names == NULL: structure only */
static int parse_container(const uint8_t *in, uint64_t len, const std::vector<std::string> *names, Container &c) {
    if (!in || len < 40) return CBCG_ERR_FORMAT;
    if (rd32(in) != CBCG_MAGIC || rd32(in + 4) != CBCG_VERSION) return CBCG_ERR_FORMAT;
    c.max_len = rd32(in + 8); c.L = rd32(in + 12); c.n_reads = rd64(in + 16);
    c.n_blocks = rd32(in + 24); c.n_chr = rd32(in + 28); c.block_reads = rd32(in + 32);
    const uint32_t mode = rd32(in + 36);
    c.gen_mode = mode & CBCG_MODE_GEN_MASK; c.fixed_len = (mode & CBCG_MODE_FIXED_LEN) ? 1u : 0u;
    c.layout_mode = mode & CBCG_MODE_LAYOUT_MASK;
    if ((mode & ~(CBCG_MODE_GEN_MASK | CBCG_MODE_FIXED_LEN | CBCG_MODE_LAYOUT_MASK)) || (c.fixed_len && c.max_len != c.L)) return CBCG_ERR_FORMAT;
    if (c.L == 0 || c.L > CBCG_MAX_READ_LEN || c.max_len > CBCG_MAX_READ_LEN || c.n_chr > MAX_CHR || c.gen_mode > 1) return CBCG_ERR_FORMAT;
    if (c.n_reads >= 0xfffffff0ull) return CBCG_ERR_FORMAT;
    uint64_t o = 40;
    c.chr_map.assign(c.n_chr, 0xffffffffu);
    for (uint32_t k = 0; k < c.n_chr; k++) {
        if (o + 4 > len) return CBCG_ERR_FORMAT;
        const uint32_t nl = rd32(in + o); o += 4;
        if (nl >= MAX_NAME || o + nl > len) return CBCG_ERR_FORMAT;
        if (names)
            for (size_t g = 0; g < names->size(); g++)
                if ((*names)[g].size() == nl && !memcmp((*names)[g].data(), in + o, nl)) c.chr_map[k] = (uint32_t)g;
        o += nl + ((4 - (nl & 3)) & 3);
    }
    if (o + 4 > len) return CBCG_ERR_FORMAT;
    c.index_bytes = rd32(in + o); o += 4;
    c.index_off = o;
    if (o + c.index_bytes > len || (uint64_t)c.n_blocks * 4u > c.index_bytes) return CBCG_ERR_FORMAT;   /* >= 4 bytes per entry */
    c.payload_off = o + c.index_bytes;
    return 0;
}

extern "C" int cbcg_decoded_size(const uint8_t *in, uint64_t in_len, uint64_t *n_reads, uint64_t *max_seq_bytes) {
    Container c;
    if (n_reads) *n_reads = 0;
    if (max_seq_bytes) *max_seq_bytes = 0;
    const int rc = parse_container(in, in_len, nullptr, c);
    if (rc) return rc;
    if (n_reads) *n_reads = c.n_reads;
    if (max_seq_bytes) *max_seq_bytes = c.n_reads * ((uint64_t)c.max_len + 1u);
    return CBCG_OK;
}

/* CBCG_POISON_DECODE=1 (tests, bench.py's correctness step): the decoder's output buffers are the encoder's work
 * buffers (K1 left this very batch's records and edits in them), so a decoder that wrote nothing would still hand K3
 * the right answer. Filled with 0xff first, only what the decoder really wrote can come out right. */
static int poison_decode_outputs(cbcg_ctx *ctx, uint64_t reads_cap, uint64_t edits_cap) {
    const char *e = getenv("CBCG_POISON_DECODE");
    if (!e || !*e || *e == '0') return 0;
    CU(cudaMemsetAsync(ctx->recs.p, 0xff, (reads_cap + 1) * sizeof(cbcg_read_rec), ctx->st));
    CU(cudaMemsetAsync(ctx->chr_out.p, 0xff, (reads_cap + 1) * 4, ctx->st));
    CU(cudaMemsetAsync(ctx->edits.p, 0xff, (edits_cap + 64) * 2, ctx->st));
    if (ctx->seq_out.p) CU(cudaMemsetAsync(ctx->seq_out.p, 0xff, ctx->seq_out.cap, ctx->st));
    return 0;
}

/* K2 decode of ctx->hblocks[0..nb) (n_reads, chr, base_pos, n_edits, payload_bytes filled in) whose payload
 * bytes lie back to back in ctx->payload. Leaves recs / edits / chr_out on the device. */
static int run_decode_blocks(cbcg_ctx *ctx, uint64_t nb, uint32_t L, int legacy, bool primed, bool fixed, uint64_t reads_cap, uint64_t edits_cap,
                             uint64_t *n_reads_out, uint64_t *n_edits_out) {
    TRY(ensure(ctx, ctx->blocks, (nb + 1) * sizeof(BlockDesc)));
    CU(cudaMemcpyAsync(ctx->blocks.p, ctx->hblocks, nb * sizeof(BlockDesc), cudaMemcpyHostToDevice, ctx->st));
    TRY(ensure(ctx, ctx->recs, (reads_cap + 1) * sizeof(cbcg_read_rec)));
    TRY(ensure(ctx, ctx->chr_out, (reads_cap + 1) * 4));
    TRY(ensure(ctx, ctx->edits, (edits_cap + 64) * 2));
    if (!legacy) primed = true;                             /* blocked containers: every block starts from a snapshot */
    const uint64_t ws_cap = legacy ? coder_ws_bytes_bound(L ? L : CBCG_MAX_READ_LEN, reads_cap, 0xffffffffull, 1, 1, 0)
                                   : coder_ws_bytes_bound(L, reads_cap, edits_cap, nb, 0, 1);
    TRY(ensure(ctx, ctx->ws, ws_cap));
    if (!legacy) TRY(ensure_fin(ctx, nb));
    TRY(reset_words(ctx));
    TRY(poison_decode_outputs(ctx, reads_cap, edits_cap));
    CoderParams p = coder_params(ctx, (uint32_t)nb, L, legacy, 1);
    p.chr = ctx->chr_out.as<uint32_t>();
    p.payload = ctx->payload.as<uint8_t>();
    p.lean = legacy ? 0u : 1u; p.short_flush = legacy ? 0u : 1u; p.primed = primed ? 1u : 0u; p.fixed_len = fixed ? 1u : 0u;
    if (launch_plan(p, (uint32_t)reads_cap, edits_cap, ws_cap, ~0ull, wptr<uint64_t>(ctx, W_OFF(totals)), ctx->st))
        return fail(ctx, CBCG_ERR_CUDA, "plan launch failed");
    ctx->stats.kernel_launches++;
    if (legacy) { ctx->gens.clear(); ctx->gens.push_back({ 0u, 1u }); }
    TRY(run_coder_generations(ctx, p, nb, primed));
    CU(cudaMemcpyAsync(ctx->hblocks, ctx->blocks.p, nb * sizeof(BlockDesc), cudaMemcpyDeviceToHost, ctx->st));
    TRY(fetch_words(ctx));
    TRY(device_error(ctx, "block decoder"));
    uint64_t nr = 0, ne = 0;
    for (uint64_t k = 0; k < nb; k++) { nr += ctx->hblocks[k].n_reads; ne += ctx->hblocks[k].n_edits; }
    *n_reads_out = nr; *n_edits_out = ne;
    return 0;
}

/* K3's reference window from the block index (ctx->hblocks, nb > 1 blocks of a blocked container): the distance between
 * the first reads of consecutive blocks of a chromosome, per read, for a tile of 128 reads, twice over, plus a read. */
static uint32_t ref_window_from_blocks(const cbcg_ctx *ctx, uint32_t max_len) {
    const uint64_t nb = ctx->gens.empty() ? 0 : (uint64_t)ctx->gens.back().first + ctx->gens.back().second;   /* blocks of the last cut / index */
    if (nb < 2 || !ctx->hblocks) return 0u;
    uint64_t span = 0, reads = 0;
    for (uint64_t k = 0; k + 1 < nb; k++) {
        const BlockDesc &a = ctx->hblocks[k], &z = ctx->hblocks[k + 1];
        if (a.chr == z.chr && z.base_pos >= a.base_pos && z.first_read > a.first_read) { span += z.base_pos - a.base_pos; reads += z.first_read - a.first_read; }
    }
    if (!reads) return 0u;
    const double want = (double)span / (double)reads * 128.0 * 2.0 + max_len + 64.0;
    return want > 1e9 ? 0u : (uint32_t)want;
}
/* fixed_len != 0: every record is that long (CBCG_MODE_FIXED_LEN container, or checked by the caller). */
static int run_reconstruct(cbcg_ctx *ctx, uint64_t n_reads, uint32_t max_len, uint32_t fixed_len, const uint32_t *chr_dev, uint32_t ref_cap_hint = 0,
                           const cbcg_read_rec *recs_dev = nullptr) {
    const uint64_t out_cap = n_reads * ((uint64_t)max_len + 1u);
    TRY(ensure(ctx, ctx->seq_out, out_cap + 64));
    TRY(ensure(ctx, ctx->tile_desc, (reconstruct_num_tiles(n_reads) + 1) * 8));
    CU(cudaMemsetAsync(wptr<unsigned long long>(ctx, W_OFF(err)), 0, 8, ctx->st));
    if (launch_reconstruct(n_reads, recs_dev ? recs_dev : ctx->recs.as<cbcg_read_rec>(), chr_dev, ctx->edits.as<uint16_t>(), ctx->dg,
                           ctx->seq_out.as<uint8_t>(), out_cap, max_len, fixed_len, ctx->tile_desc.as<uint64_t>(),
                           wptr<uint32_t>(ctx, W_OFF(ticket)), wptr<uint64_t>(ctx, W_OFF(total_bytes)),
                           wptr<unsigned long long>(ctx, W_OFF(err)), ctx->st, ctx->kev[2], ctx->kev[3], ref_cap_hint))
        return fail(ctx, CBCG_ERR_CUDA, "K3 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    ctx->stats.kernel_launches++;
    return 0;
}

/* index entries of a parsed container -> ctx->hblocks */
static int blocks_from_index(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, const Container &c,
                             uint64_t *reads_total, uint64_t *edits_total, uint64_t *payload_total) {
    TRY(ensure_hblocks(ctx, (size_t)c.n_blocks + 1));
    uint64_t nr = 0, ne = 0, pb = 0;
    IndexState st = index_state(c.block_reads);
    uint64_t o = c.index_off;
    uint32_t prev_gen = 0;
    for (uint32_t k = 0; k < c.n_blocks; k++) {
        BlockDesc &b = ctx->hblocks[k];
        if (!index_get(in, c.index_off + c.index_bytes, o, st, b, c.layout_mode)) return fail(ctx, CBCG_ERR_FORMAT, "block index entry %u malformed", k);
        const uint32_t chr = b.chr;
        if (chr >= c.n_chr) return fail(ctx, CBCG_ERR_FORMAT, "block %u names chromosome %u of %u", k, chr, c.n_chr);
        if (c.chr_map[chr] == 0xffffffffu) return fail(ctx, CBCG_ERR_NO_REFERENCE, "block %u: chromosome not in the loaded reference", k);
        if (b.gen < prev_gen || (c.gen_mode == 0 && b.gen != 0)) return fail(ctx, CBCG_ERR_FORMAT, "block %u: bad generation %u", k, b.gen);
        prev_gen = b.gen;
        b.chr = c.chr_map[chr];
        nr += b.n_reads; ne += b.n_edits; pb += b.payload_bytes;
    }
    gens_from_blocks(ctx, c.n_blocks);
    if (nr != c.n_reads) return fail(ctx, CBCG_ERR_FORMAT, "index holds %llu reads, header says %llu", (unsigned long long)nr, (unsigned long long)c.n_reads);
    if (c.payload_off + pb > in_len) return fail(ctx, CBCG_ERR_FORMAT, "payload truncated");
    *reads_total = nr; *edits_total = ne; *payload_total = pb;
    return 0;
}

/* Shared by cbcg_decode / cbcg_decode_edits: container (or legacy stream) -> recs/edits/chr on the device. */
static int decode_to_records(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                             uint64_t *n_reads, uint64_t *n_edits, uint32_t *max_len, uint32_t *fixed_len) {
    *fixed_len = 0;
    if (!ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "cbcg_set_reference has not been called");
    CU(cudaSetDevice(ctx->device));
    set_carveout_all(-1);
    ctx->have_decoded = false;
    ctx->have_encoded = false;                              /* ctx->payload and ctx->hblocks are about to hold another container */
    cbcg_stats &S = ctx->stats;
    S = cbcg_stats();
    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    if (!legacy) {
        Container c;
        int rc = parse_container(in, in_len, &ctx->names, c);
        if (rc) return fail(ctx, rc, "malformed container header");
        uint64_t nr = 0, ne = 0, pb = 0;
        ctx->layout_mode = c.layout_mode;
        TRY(blocks_from_index(ctx, in, in_len, c, &nr, &ne, &pb));
        *max_len = c.max_len ? c.max_len : 1;
        *fixed_len = c.fixed_len ? c.L : 0u;
        *n_reads = 0; *n_edits = 0;
        if (c.n_blocks == 0) return 0;
        TRY(ensure(ctx, ctx->payload, pb + 64));
        if (pb) CU(cudaMemcpyAsync(ctx->payload.p, in + c.payload_off, pb, cudaMemcpyHostToDevice, ctx->st));
        S.h2d_bytes = pb + (uint64_t)c.n_blocks * sizeof(BlockDesc);
        CU(cudaEventRecord(ctx->ev[1], ctx->st));
        TRY(run_decode_blocks(ctx, c.n_blocks, c.L, 0, c.gen_mode == 1, c.fixed_len != 0, nr, ne, n_reads, n_edits));
        S.n_blocks = c.n_blocks;
    } else {
        if (!in || in_len < 4) return fail(ctx, CBCG_ERR_FORMAT, "legacy stream too short");
        if (in_len > 0xfffffff0ull) return fail(ctx, CBCG_ERR_ARG, "legacy stream too large");
        TRY(ensure(ctx, ctx->payload, in_len + 64));
        CU(cudaMemcpyAsync(ctx->payload.p, in, in_len, cudaMemcpyHostToDevice, ctx->st));
        S.h2d_bytes = in_len;
        CU(cudaEventRecord(ctx->ev[1], ctx->st));
        /* the read count is not in the stream: decode into a guessed capacity, double on overflow */
        uint64_t reads_cap = std::max<uint64_t>(in_len * 2, 1u << 16);
        for (;;) {
            TRY(ensure_hblocks(ctx, 2));
            BlockDesc &b = ctx->hblocks[0];
            memset(&b, 0, sizeof b);
            b.n_reads = (uint32_t)std::min<uint64_t>(reads_cap, 0xfffffff0ull);
            b.n_edits = (uint32_t)std::min<uint64_t>(reads_cap * 4, 0xfffffff0ull);
            b.payload_bytes = (uint32_t)in_len;
            int rc = run_decode_blocks(ctx, 1, 0, 1, false, false, b.n_reads, b.n_edits, n_reads, n_edits);
            if (rc == CBCG_ERR_CAPACITY && reads_cap < (1ull << 31)) { reads_cap *= 4; continue; }
            if (rc) return rc;
            break;
        }
        *max_len = ctx->hblocks[0].pad;                     /* header read length (src/sam_file_allocation.c:365) */
        S.n_blocks = 1;
    }
    CU(cudaEventRecord(ctx->ev[2], ctx->st));
    S.n_reads = *n_reads; S.n_edits = *n_edits;
    return 0;
}

/* ------------------------------------------------------------------------------------------------ pipelined decode
 * cbcg_decode of a large container of equal-length reads: the last generation is decoded group by group on side
 * streams, each group followed by its own K3 launch and its own device -> host copy (output offsets are closed-form),
 * so text is on the PCIe link while other groups are still being decoded. Containers written by the pipelined encoder
 * have their small blocks at the end of the batch: those groups finish first. */
static int decode_pipelined(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, uint8_t *seq_out, uint64_t seq_cap,
                            uint64_t *seq_len, uint64_t *n_reads) {
    Container c;
    if (parse_container(in, in_len, &ctx->names, c)) return PIPE_FALLBACK;         /* the one-stream path reports it */
    if (!c.fixed_len || c.gen_mode != 1 || c.n_reads < pipe_min_reads() || !ctx->dg.n_chr || !seq_out) return PIPE_FALLBACK;
    const uint64_t line = (uint64_t)c.L + 1u, bytes = c.n_reads * line;
    if (bytes > seq_cap) return PIPE_FALLBACK;
    TRY(pipe_init(ctx));
    set_carveout_all(100);
    ctx->have_decoded = false;
    ctx->have_encoded = false;                              /* ctx->payload and ctx->hblocks are about to hold another container */
    cbcg_stats &S = ctx->stats;
    S = cbcg_stats();
    uint64_t nr = 0, ne = 0, pb = 0;
    ctx->layout_mode = c.layout_mode;
    TRY(blocks_from_index(ctx, in, in_len, c, &nr, &ne, &pb));
    if (ctx->gens.size() < 2) return PIPE_FALLBACK;
    const uint32_t nb = c.n_blocks;
    BlockDesc *hb = ctx->hblocks;
    const uint32_t k3_ref_cap = ref_window_from_blocks(ctx, c.L);
    const uint32_t last_first = ctx->gens.back().first, last_n = ctx->gens.back().second;
    uint64_t early_reads = 0;
    for (uint32_t k = 0; k < last_first; k++) early_reads += hb[k].n_reads;
    /* groups of last-generation blocks: the size classes the encoder's ramp left (blocks of one class end together),
       else about equal read counts */
    uint32_t gb[PIPE_CHUNKS + 1]; uint64_t gr[PIPE_CHUNKS + 1];
    gb[0] = last_first; gr[0] = early_reads;
    bool by_class = false;
    {
        uint32_t marks[PIPE_CHUNKS + 1], nm = 0, ref_size = hb[last_first].n_reads;
        for (uint32_t k = last_first + 1; k + 1 < last_first + last_n && nm <= PIPE_CHUNKS; k++) {
            const uint32_t sz = hb[k].n_reads;
            if (hb[k].chr == hb[k - 1].chr && (sz * 20u > ref_size * 21u || sz * 21u < ref_size * 20u) && sz == hb[k + 1].n_reads) {
                if (nm < PIPE_CHUNKS + 1) marks[nm] = k;
                nm++; ref_size = sz;
            }
        }
        if (nm >= 1 && nm <= PIPE_CHUNKS - 1) {
            uint64_t r = early_reads; uint32_t k = last_first, g = 1;
            for (; g <= PIPE_CHUNKS; g++) {
                const uint32_t stop = (g <= nm) ? last_first + ((marks[g - 1] - last_first + 3u) & ~3u) : last_first + last_n;   /* whole CTAs */
                while (k < stop && k < last_first + last_n) r += hb[k++].n_reads;
                gb[g] = k; gr[g] = r;
            }
            by_class = true;
        }
    }
    if (!by_class) {
        uint32_t k = last_first; uint64_t r = early_reads;
        for (uint32_t g = 1; g <= PIPE_CHUNKS; g++) {
            const uint64_t want = early_reads + (nr - early_reads) * g / PIPE_CHUNKS;
            while (k < last_first + last_n && (r < want || g == PIPE_CHUNKS || ((k - last_first) & 3u))) r += hb[k++].n_reads;   /* whole CTAs */
            gb[g] = k; gr[g] = r;
        }
    }
    TRY(ensure(ctx, ctx->payload, pb + 96));
    TRY(ensure(ctx, ctx->blocks, ((uint64_t)nb + 1) * sizeof(BlockDesc)));
    TRY(ensure(ctx, ctx->recs, (nr + 1) * sizeof(cbcg_read_rec)));
    TRY(ensure(ctx, ctx->chr_out, (nr + 1) * 4));
    TRY(ensure(ctx, ctx->edits, (ne + 64) * 2));
    const uint64_t ws_cap = coder_ws_bytes_bound(c.L, nr, ne, nb, 0, 1);
    TRY(ensure(ctx, ctx->ws, ws_cap));
    TRY(ensure_fin(ctx, nb));
    TRY(ensure(ctx, ctx->seq_out, bytes + 64));
    TRY(ensure(ctx, ctx->tile_desc, (reconstruct_num_tiles(nr) + 1) * 8));

    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    /* the container and the descriptors come in by kernels when the caller's buffer is pinned (read in place over PCIe:
       the host -> device copy engine may be busy with another batch's input); the payload keeps the misalignment it has in
       the caller's buffer, the coder reads it byte by byte */
    uint32_t pay_shift = 0;
    if (pb && host_mapped(in)) {
        const uint8_t *src = in + c.payload_off;
        pay_shift = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 15u);
        const uint64_t body = (pb + pay_shift) & ~15ull, tail = pb + pay_shift - body;     /* nothing is read past the caller's last byte */
        if (launch_copy16(ctx->payload.p, src - pay_shift, body, ctx->st) ||
            launch_d2h_bytes(ctx->payload.as<uint8_t>() + body, src - pay_shift + body, tail, ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "payload copy launch failed");
    } else if (pb) CU(cudaMemcpyAsync(ctx->payload.p, in + c.payload_off, pb, cudaMemcpyHostToDevice, ctx->st));
    if (launch_copy16(ctx->blocks.p, hb, (uint64_t)nb * sizeof(BlockDesc), ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "descriptor copy launch failed");
    TRY(reset_words(ctx));
    TRY(poison_decode_outputs(ctx, nr, ne));
    CoderParams p = coder_params(ctx, nb, c.L, 0, 1);
    p.chr = ctx->chr_out.as<uint32_t>();
    p.payload = ctx->payload.as<uint8_t>() + pay_shift;
    p.lean = 1u; p.short_flush = 1u; p.primed = 1u; p.fixed_len = 1u;
    if (launch_plan(p, (uint32_t)nr, ne, ws_cap, ~0ull, wptr<uint64_t>(ctx, W_OFF(totals)), ctx->st))
        return fail(ctx, CBCG_ERR_CUDA, "plan launch failed");
    S.kernel_launches++;
    uint8_t *snap = nullptr;
    TRY(run_early_generations(ctx, p, &snap));
    for (uint32_t g = 0; g <= PIPE_CHUNKS; g++) {            /* g = 0: the reads of the early generations */
        const uint64_t r0 = g ? gr[g - 1] : 0, r1 = g ? gr[g] : early_reads;
        /* the early generations' reads are rebuilt on the main stream BEFORE the last generation is launched: once its
           CTAs hold every SM, a K3 CTA finds room only when one of them retires */
        cudaStream_t sd = g ? ctx->ps[g % PIPE_MAX] : ctx->st;
        if (g) CU(cudaStreamWaitEvent(sd, ctx->kev2[0], 0));
        if (g && gb[g] > gb[g - 1]) {
            CoderParams q = p;
            q.block_begin = gb[g - 1]; q.n_blocks = gb[g] - gb[g - 1]; q.snap = snap; q.n_sub = gen_n_sub(ctx, q.block_begin);
            if (launch_coder(q, sd)) return fail(ctx, CBCG_ERR_CUDA, "K2 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
            S.kernel_launches += coder_launches(q);
        }
        CU(cudaEventRecord(ctx->tev[2 * g], sd));
        if (r1 > r0) {
            if (launch_reconstruct(r1 - r0, ctx->recs.as<cbcg_read_rec>() + r0, ctx->chr_out.as<uint32_t>() + r0, ctx->edits.as<uint16_t>(),
                                   ctx->dg, ctx->seq_out.as<uint8_t>() + r0 * line, (r1 - r0) * line, c.L, c.L, ctx->tile_desc.as<uint64_t>(),
                                   wptr<uint32_t>(ctx, W_OFF(ticket)), wptr<uint64_t>(ctx, W_OFF(total_bytes)),
                                   wptr<unsigned long long>(ctx, W_OFF(err)), sd, nullptr, nullptr, k3_ref_cap))
                return fail(ctx, CBCG_ERR_CUDA, "K3 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
            S.kernel_launches++;
            CU(cudaEventRecord(ctx->tev[2 * g + 1], sd));
            if (!g) {                                        /* its copy rides a side stream; the groups start behind the K3 launch */
                CU(cudaEventRecord(ctx->kev2[0], ctx->st));
                sd = ctx->ps[0];
                CU(cudaStreamWaitEvent(sd, ctx->kev2[0], 0));
                CU(cudaMemcpyAsync(seq_out + r0 * line, ctx->seq_out.as<uint8_t>() + r0 * line, (r1 - r0) * line, cudaMemcpyDeviceToHost, sd));
            }
        } else if (!g) CU(cudaEventRecord(ctx->kev2[0], ctx->st));
        if (!g) CU(cudaEventRecord(ctx->dev2[0], sd));
    }
    /* The groups' texts go out on ONE stream, in the order the groups are expected to finish (smallest blocks first).
       Issued per group stream, the copy engine served them in an order of its own: the group that was ready first
       (6.3 ms) was copied fourth (trace, config 2), and the engine idled until the second group was ready. */
    {
        uint32_t order[PIPE_CHUNKS]; uint32_t no = 0;
        for (uint32_t g = 1; g <= PIPE_CHUNKS; g++) if (gr[g] > gr[g - 1]) order[no++] = g;
        std::stable_sort(order, order + no, [&](uint32_t a, uint32_t b) {
            const uint32_t sa = gb[a] > gb[a - 1] ? hb[gb[a - 1]].n_reads : 0u, sb2 = gb[b] > gb[b - 1] ? hb[gb[b - 1]].n_reads : 0u;
            return sa < sb2;
        });
        CU(cudaStreamWaitEvent(ctx->cs, ctx->dev2[0], 0));   /* behind the early generations' text */
        for (uint32_t k = 0; k < no; k++) {
            const uint32_t g = order[k];
            const uint64_t r0 = gr[g - 1], r1 = gr[g];
            CU(cudaStreamWaitEvent(ctx->cs, ctx->tev[2 * g + 1], 0));
            CU(cudaMemcpyAsync(seq_out + r0 * line, ctx->seq_out.as<uint8_t>() + r0 * line, (r1 - r0) * line, cudaMemcpyDeviceToHost, ctx->cs));
            CU(cudaEventRecord(ctx->dev2[g], ctx->cs));
        }
        for (uint32_t g = 1; g <= PIPE_CHUNKS; g++) if (gr[g] <= gr[g - 1]) CU(cudaEventRecord(ctx->dev2[g], ctx->ps[g % PIPE_MAX]));
    }
    for (uint32_t g = 0; g <= PIPE_CHUNKS; g++) CU(cudaStreamWaitEvent(ctx->st, ctx->dev2[g], 0));
    CU(cudaEventRecord(ctx->ev[1], ctx->st));
    if (launch_copy16(ctx->hblocks, ctx->blocks.p, (uint64_t)nb * sizeof(BlockDesc), ctx->st)) return fail(ctx, CBCG_ERR_CUDA, "descriptor copy launch failed");
    TRY(fetch_words(ctx));
    TRY(device_error(ctx, "pipelined decode"));
    uint64_t got_r = 0, got_e = 0;
    for (uint32_t k = 0; k < nb; k++) { got_r += hb[k].n_reads; got_e += hb[k].n_edits; }
    if (got_r != nr) return fail(ctx, CBCG_ERR_CORRUPT, "decoded %llu reads, the index says %llu", (unsigned long long)got_r, (unsigned long long)nr);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[1]);
    if (getenv("CBCG_PIPE_TRACE")) {
        float t0 = 0; cudaEventElapsedTime(&t0, ctx->ev[0], ctx->kev2[0]);
        fprintf(stderr, "[cbcg pipe dec] early generations done %.2f ms\n", t0);
        for (uint32_t g = 0; g <= PIPE_CHUNKS; g++) {
            float d = 0, k2 = 0, k3 = 0; cudaEventElapsedTime(&d, ctx->ev[0], ctx->dev2[g]);
            cudaEventElapsedTime(&k2, ctx->ev[0], ctx->tev[2 * g]); cudaEventElapsedTime(&k3, ctx->ev[0], ctx->tev[2 * g + 1]);
            fprintf(stderr, "[cbcg pipe dec] group %u blocks %u reads %llu: decoded %.2f ms, rebuilt %.2f ms, text on the host %.2f ms\n", g,
                    g ? gb[g] - gb[g - 1] : last_first, (unsigned long long)(g ? gr[g] - gr[g - 1] : early_reads), k2, k3, d);
        }
        fprintf(stderr, "[cbcg pipe dec] all %.2f ms\n", S.ms_total);
    }
    S.h2d_bytes = pb + (uint64_t)nb * sizeof(BlockDesc); S.d2h_bytes = bytes;
    S.n_reads = nr; S.n_edits = got_e; S.n_blocks = nb;
    *seq_len = bytes; if (n_reads) *n_reads = nr;
    ctx->dec_bytes = bytes; ctx->dec_n_reads = nr; ctx->have_decoded = true;
    return CBCG_OK;
}

extern "C" int cbcg_decode(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                           uint8_t *seq_out, uint64_t seq_cap, uint64_t *seq_len, uint64_t *n_reads) {
    if (!ctx || !seq_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_decode: bad argument");
    uint64_t nr = 0, ne = 0; uint32_t max_len = 1, fixed_len = 0;
    *seq_len = 0; if (n_reads) *n_reads = 0;
    if (!legacy) {
        CU(cudaSetDevice(ctx->device));
        const int rc = decode_pipelined(ctx, in, in_len, seq_out, seq_cap, seq_len, n_reads);
        if (rc < 0) pipe_drain(ctx);                         /* copies into seq_out may still be queued */
        if (rc != PIPE_FALLBACK) return rc;
    }
    TRY(decode_to_records(ctx, in, in_len, legacy, &nr, &ne, &max_len, &fixed_len));
    if (n_reads) *n_reads = nr;
    if (!nr) return CBCG_OK;
    if (legacy) max_len = CBCG_MAX_READ_LEN;                /* per-read lengths are coded mod 256 (src/read_compression.c:29-33) */
    TRY(run_reconstruct(ctx, nr, max_len, fixed_len, ctx->chr_out.as<uint32_t>(), legacy ? 0u : ref_window_from_blocks(ctx, max_len)));
    CU(cudaEventRecord(ctx->ev[3], ctx->st));
    TRY(fetch_words(ctx));
    TRY(device_error(ctx, "read reconstruction"));
    cudaEventElapsedTime(&ctx->stats.ms_k3, ctx->kev[2], ctx->kev[3]);
    const uint64_t bytes = ctx->hw->total_bytes;
    *seq_len = bytes;
    ctx->dec_bytes = bytes; ctx->dec_n_reads = nr; ctx->have_decoded = true;
    cbcg_stats &S = ctx->stats;
    cudaEventElapsedTime(&S.ms_h2d, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&S.ms_code, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&S.ms_reconstruct, ctx->ev[2], ctx->ev[3]);
    if (bytes > seq_cap || !seq_out) return fail(ctx, CBCG_ERR_CAPACITY, "decoded text is %llu bytes, room for %llu", (unsigned long long)bytes, (unsigned long long)seq_cap);
    CU(cudaEventRecord(ctx->ev[4], ctx->st));
    CU(cudaMemcpyAsync(seq_out, ctx->seq_out.p, bytes, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaEventRecord(ctx->ev[5], ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    cudaEventElapsedTime(&S.ms_d2h, ctx->ev[4], ctx->ev[5]);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[5]);
    S.d2h_bytes = bytes;
    return CBCG_OK;
}

extern "C" int cbcg_decode_edits(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                                 cbcg_read_rec *recs, uint64_t recs_cap, uint32_t *chr, uint16_t *edits,
                                 uint64_t edits_cap, uint64_t *n_reads, uint64_t *n_edits) {
    if (!ctx || !n_reads || !n_edits) return fail(ctx, CBCG_ERR_ARG, "cbcg_decode_edits: bad argument");
    uint64_t nr = 0, ne = 0; uint32_t max_len = 1, fixed_len = 0;
    *n_reads = 0; *n_edits = 0;
    TRY(decode_to_records(ctx, in, in_len, legacy, &nr, &ne, &max_len, &fixed_len));
    *n_reads = nr; *n_edits = ne;
    if (nr > recs_cap || ne > edits_cap) return fail(ctx, CBCG_ERR_CAPACITY, "%llu reads / %llu edits decoded, room for %llu / %llu",
                                                     (unsigned long long)nr, (unsigned long long)ne, (unsigned long long)recs_cap, (unsigned long long)edits_cap);
    /* blocks were decoded into disjoint [first_read, +n_reads) / [edit_base, +n_edits) ranges that are dense
       because the index carries exact counts (legacy: one block) */
    if (nr && recs) CU(cudaMemcpyAsync(recs, ctx->recs.p, nr * sizeof(cbcg_read_rec), cudaMemcpyDeviceToHost, ctx->st));
    if (nr && chr) CU(cudaMemcpyAsync(chr, ctx->chr_out.p, nr * 4, cudaMemcpyDeviceToHost, ctx->st));
    if (ne && edits) CU(cudaMemcpyAsync(edits, ctx->edits.p, ne * 2, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ region decode
 * cbcg_region_plan / cbcg_decode_region (DESIGN.md, "Region decode"). The blocks of generation g start from the snapshot
 * that merges every block of the generations before g, so the blocks a query touches are decoded after every block of
 * every generation before the latest touched one (g*), and of g* only the touched blocks are. One host routine walks the
 * header and the index once and returns that selection; the decode hands it to the block decoder as a reduced descriptor
 * table (each block keeps its generation, the FLAG target comes from the whole index), K5 keeps the reads that overlap
 * a region and K3 rebuilds only those. */
static int check_regions(cbcg_ctx *ctx, const cbcg_region *regions, uint32_t n_regions) {
    if (!regions || !n_regions) return fail(ctx, CBCG_ERR_ARG, "no regions");
    for (uint32_t k = 0; k < n_regions; k++)
        if (!regions[k].name || regions[k].start == 0 || regions[k].start > regions[k].end)
            return fail(ctx, CBCG_ERR_ARG, "region %u: NULL name, start 0 or start > end", k);
    return 0;
}
/* sorted by (chr, start), overlapping or adjacent intervals merged: their ends ascend too */
static void merge_intervals(std::vector<RegionIv> &iv) {
    std::sort(iv.begin(), iv.end(), [](const RegionIv &a, const RegionIv &b) { return a.chr != b.chr ? a.chr < b.chr : a.start < b.start; });
    size_t n = 0;
    for (size_t k = 0; k < iv.size(); k++) {
        if (n && iv[n - 1].chr == iv[k].chr && (iv[n - 1].end == UINT64_MAX || iv[k].start <= iv[n - 1].end + 1)) {
            iv[n - 1].end = std::max(iv[n - 1].end, iv[k].end);
            continue;
        }
        iv[n++] = iv[k];
    }
    iv.resize(n);
}
/* the regions whose name is in `names`, by ordinal into it; other names match nothing */
static std::vector<RegionIv> region_intervals(const cbcg_region *regions, uint32_t n_regions, const std::vector<std::string> &names) {
    std::vector<RegionIv> iv;
    for (uint32_t k = 0; k < n_regions; k++) {
        const size_t nl = strlen(regions[k].name);
        for (size_t g = 0; g < names.size(); g++)
            if (names[g].size() == nl && !memcmp(names[g].data(), regions[k].name, nl)) { iv.push_back({ (uint32_t)g, 0u, regions[k].start, regions[k].end }); break; }
    }
    merge_intervals(iv);
    return iv;
}

/* the chromosome table of a parsed container */
static std::vector<std::string> container_names(const uint8_t *in, const Container &c) {
    std::vector<std::string> names(c.n_chr);
    for (uint64_t o = 40, k = 0; k < c.n_chr; k++) {                 /* parse_container has checked the name table */
        const uint32_t nl = rd32(in + o); o += 4;
        names[k].assign(reinterpret_cast<const char *>(in + o), nl);
        o += nl + ((4 - (nl & 3)) & 3);
    }
    return names;
}

struct RegionPlan {
    Container c;
    std::vector<BlockDesc> blocks;             /* the whole index (container chromosome ordinals); first_read / payload_off within the container */
    std::vector<uint32_t> sel;                 /* blocks to decode, ascending */
    std::vector<RegionIv> iv;                  /* the regions by container chromosome ordinal */
    uint32_t max_block_reads = 0;              /* longest block of the whole index: the FLAG target of the merged snapshots */
    uint64_t n_reads = 0, n_edits = 0, payload_bytes = 0, max_seq_bytes = 0;
};

/* Header + index -> the blocks to decode. A block's reads start within [its base_pos, the next block's base_pos on the same
 * chromosome] (no upper bound for a chromosome's last block), and a read that starts up to max_len + 255 bases before a
 * region (<= 255 deletions per read) can still reach into it: the selection is generous, K5 is exact. Reads no payload. */
static int plan_region(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, const cbcg_region *regions, uint32_t n_regions, RegionPlan &P,
                       const std::vector<std::string> *genome = nullptr) {   /* genome: fills P.c.chr_map */
    TRY(check_regions(ctx, regions, n_regions));
    Container &c = P.c;
    if (parse_container(in, in_len, genome, c)) return fail(ctx, CBCG_ERR_FORMAT, "malformed container header");
    P.iv = region_intervals(regions, n_regions, container_names(in, c));
    P.blocks.resize(c.n_blocks);
    IndexState st = index_state(c.block_reads);
    uint64_t o = c.index_off, first = 0, pay = 0;
    uint32_t prev_gen = 0;
    for (uint32_t k = 0; k < c.n_blocks; k++) {
        BlockDesc &b = P.blocks[k];
        if (!index_get(in, c.index_off + c.index_bytes, o, st, b, c.layout_mode)) return fail(ctx, CBCG_ERR_FORMAT, "block index entry %u malformed", k);
        if (b.chr >= c.n_chr) return fail(ctx, CBCG_ERR_FORMAT, "block %u names chromosome %u of %u", k, b.chr, c.n_chr);
        if (b.gen < prev_gen || (c.gen_mode == 0 && b.gen != 0)) return fail(ctx, CBCG_ERR_FORMAT, "block %u: bad generation %u", k, b.gen);
        prev_gen = b.gen;
        b.first_read = (uint32_t)first; b.payload_off = pay;
        first += b.n_reads; pay += b.payload_bytes;
        P.max_block_reads = std::max(P.max_block_reads, b.n_reads);
    }
    if (first != c.n_reads) return fail(ctx, CBCG_ERR_FORMAT, "index holds %llu reads, header says %llu", (unsigned long long)first, (unsigned long long)c.n_reads);
    if (c.payload_off + pay > in_len) return fail(ctx, CBCG_ERR_FORMAT, "payload truncated");
    const uint64_t reach = (uint64_t)c.max_len + 255u;
    std::vector<uint8_t> touched(c.n_blocks, 0);
    bool any = false;
    uint32_t g_star = 0;
    for (uint32_t k = 0; k < c.n_blocks; k++) {
        const BlockDesc &b = P.blocks[k];
        const uint64_t lo = b.base_pos;
        const uint64_t hi = (k + 1 < c.n_blocks && P.blocks[k + 1].chr == b.chr) ? P.blocks[k + 1].base_pos : UINT64_MAX;
        /* the first interval of this chromosome that ends at or after lo: the only one that can start too early to matter */
        const auto it = std::lower_bound(P.iv.begin(), P.iv.end(), b, [&](const RegionIv &v, const BlockDesc &) {
            return v.chr < b.chr || (v.chr == b.chr && v.end < lo); });
        if (it == P.iv.end() || it->chr != b.chr) continue;
        if (hi != UINT64_MAX && hi + reach <= it->start) continue;
        touched[k] = 1; any = true; g_star = std::max(g_star, b.gen);
    }
    uint64_t touched_reads = 0;
    for (uint32_t k = 0; any && k < c.n_blocks; k++) {
        const BlockDesc &b = P.blocks[k];
        if (b.gen > g_star || (b.gen == g_star && !touched[k])) continue;
        P.sel.push_back(k);
        P.n_reads += b.n_reads; P.n_edits += b.n_edits; P.payload_bytes += b.payload_bytes;
        if (touched[k]) touched_reads += b.n_reads;
    }
    P.max_seq_bytes = touched_reads * ((uint64_t)c.max_len + 1u);
    return 0;
}

extern "C" int cbcg_region_plan(const uint8_t *in, uint64_t in_len, int legacy, const cbcg_region *regions, uint32_t n_regions,
                                uint64_t *n_blocks, uint64_t *n_reads, uint64_t *payload_bytes, uint64_t *max_seq_bytes) {
    for (uint64_t *p : { n_blocks, n_reads, payload_bytes, max_seq_bytes }) if (p) *p = 0;
    if (legacy) {                                            /* one block, decoded whole; the stream does not store its read count */
        TRY(check_regions(nullptr, regions, n_regions));
        if (!in || in_len < 4) return CBCG_ERR_FORMAT;
        if (n_blocks) *n_blocks = 1;
        if (n_reads) *n_reads = UINT64_MAX;
        if (payload_bytes) *payload_bytes = in_len;
        if (max_seq_bytes) *max_seq_bytes = UINT64_MAX;
        return CBCG_OK;
    }
    RegionPlan P;
    TRY(plan_region(nullptr, in, in_len, regions, n_regions, P));
    if (n_blocks) *n_blocks = P.sel.size();
    if (n_reads) *n_reads = P.n_reads;
    if (payload_bytes) *payload_bytes = P.payload_bytes;
    if (max_seq_bytes) *max_seq_bytes = P.max_seq_bytes;
    return CBCG_OK;
}

/* K5 over the nr decoded records in ctx->recs / ctx->chr_out: the kept reads -> ctx->sel_*, *n_sel their number */
static int run_region_select(cbcg_ctx *ctx, uint64_t nr, const std::vector<RegionIv> &iv, const std::vector<uint64_t> &runs, uint64_t *n_sel) {
    *n_sel = 0;
    const uint64_t iv_bytes = iv.size() * sizeof(RegionIv);
    TRY(ensure(ctx, ctx->reg, iv_bytes + runs.size() * 8 + 64));
    TRY(ensure(ctx, ctx->sel_recs, (nr + 1) * sizeof(cbcg_read_rec)));
    TRY(ensure(ctx, ctx->sel_chr, (nr + 1) * 4));
    TRY(ensure(ctx, ctx->sel_ids, (nr + 1) * 8));
    TRY(ensure(ctx, ctx->tile_desc, (region_num_tiles(nr) + 1) * 8));
    CU(cudaMemcpyAsync(ctx->reg.p, iv.data(), iv_bytes, cudaMemcpyHostToDevice, ctx->st));
    const uint64_t *d_runs = reinterpret_cast<const uint64_t *>(ctx->reg.as<uint8_t>() + iv_bytes);
    CU(cudaMemcpyAsync(const_cast<uint64_t *>(d_runs), runs.data(), runs.size() * 8, cudaMemcpyHostToDevice, ctx->st));
    if (launch_region_select(nr, ctx->recs.as<cbcg_read_rec>(), ctx->chr_out.as<uint32_t>(), ctx->reg.as<RegionIv>(), (uint32_t)iv.size(),
                             d_runs, (uint32_t)(runs.size() / 2), ctx->sel_recs.as<cbcg_read_rec>(), ctx->sel_chr.as<uint32_t>(),
                             ctx->sel_ids.as<uint64_t>(), ctx->tile_desc.as<uint64_t>(), wptr<uint32_t>(ctx, W_OFF(ticket)),
                             wptr<uint64_t>(ctx, W_OFF(n_selected)), wptr<unsigned long long>(ctx, W_OFF(err)), ctx->st))
        return fail(ctx, CBCG_ERR_CUDA, "region select launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    ctx->stats.kernel_launches++;
    TRY(fetch_words(ctx));                                   /* synchronises: the host vectors may go */
    TRY(device_error(ctx, "region select"));
    *n_sel = ctx->hw->n_selected;
    return 0;
}

/* The region's reads of a container (or legacy stream) -> ctx->sel_recs / sel_chr / sel_ids (*n_sel of them), decoded as
 * cbcg_decode_region describes; *nr and *ne: the reads and edits the block decoder decoded. Events ev[0..2] are recorded. */
static int region_records(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy, const cbcg_region *regions, uint32_t n_regions,
                          uint64_t *nr_out, uint64_t *ne_out, uint64_t *n_sel_out, uint32_t *max_len_out, uint32_t *fixed_len_out) {
    TRY(check_regions(ctx, regions, n_regions));
    if (!ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "cbcg_set_reference has not been called");
    uint64_t nr = 0, ne = 0; uint32_t max_len = 1, fixed_len = 0;
    std::vector<RegionIv> iv;                                /* by genome ordinal */
    std::vector<uint64_t> runs;                              /* (dense first read, container first read) per run of consecutive blocks */
    cbcg_stats &S = ctx->stats;
    if (legacy) {                                            /* one block: decoded whole, then filtered */
        TRY(decode_to_records(ctx, in, in_len, 1, &nr, &ne, &max_len, &fixed_len));
        max_len = CBCG_MAX_READ_LEN;                         /* per-read lengths are coded mod 256 (src/read_compression.c:29-33) */
        iv = region_intervals(regions, n_regions, ctx->names);
        runs = { 0ull, 0ull };
    } else {
        RegionPlan P;
        TRY(plan_region(ctx, in, in_len, regions, n_regions, P, &ctx->names));
        const Container &c = P.c;
        const std::vector<uint32_t> &chr_map = c.chr_map;
        CU(cudaSetDevice(ctx->device));
        set_carveout_all(-1);
        ctx->have_decoded = false;
        ctx->have_encoded = false;                          /* ctx->payload and ctx->hblocks are about to hold another container */
        S = cbcg_stats();
        CU(cudaEventRecord(ctx->ev[0], ctx->st));
        /* chromosomes: only the blocks that are decoded have to be in the loaded reference */
        const uint64_t nb = P.sel.size();
        TRY(ensure_hblocks(ctx, nb + 1));
        for (uint64_t j = 0; j < nb; j++) {
            BlockDesc b = P.blocks[P.sel[j]];
            if (chr_map[b.chr] == 0xffffffffu) return fail(ctx, CBCG_ERR_NO_REFERENCE, "block %u: chromosome not in the loaded reference", P.sel[j]);
            b.chr = chr_map[b.chr];
            b.first_read = 0; b.payload_off = 0;             /* the plan kernel numbers the reduced table densely */
            ctx->hblocks[j] = b;
        }
        for (RegionIv &v : P.iv) v.chr = chr_map[v.chr];
        for (const RegionIv &v : P.iv) if (v.chr != 0xffffffffu) iv.push_back(v);
        merge_intervals(iv);
        ctx->layout_mode = c.layout_mode;
        gens_from_blocks(ctx, nb);
        ctx->max_block_reads = P.max_block_reads;           /* the encoder's FLAG target: the whole container's longest block */
        max_len = c.max_len ? c.max_len : 1;
        fixed_len = c.fixed_len ? c.L : 0u;
        /* the payload of the selection: the prefix of the early generations and one run per group of adjacent blocks */
        TRY(ensure(ctx, ctx->payload, P.payload_bytes + 64));
        uint64_t dense = 0, at = 0;
        for (uint64_t j = 0; j < nb;) {
            uint64_t e = j + 1;
            while (e < nb && P.sel[e] == P.sel[e - 1] + 1) e++;
            const BlockDesc &a = P.blocks[P.sel[j]], &z = P.blocks[P.sel[e - 1]];
            const uint64_t bytes = z.payload_off + z.payload_bytes - a.payload_off;
            if (bytes) CU(cudaMemcpyAsync(ctx->payload.as<uint8_t>() + at, in + c.payload_off + a.payload_off, bytes, cudaMemcpyHostToDevice, ctx->st));
            runs.push_back(dense); runs.push_back(a.first_read);
            at += bytes;
            for (uint64_t k = j; k < e; k++) dense += P.blocks[P.sel[k]].n_reads;
            j = e;
        }
        S.h2d_bytes = P.payload_bytes + nb * sizeof(BlockDesc);
        CU(cudaEventRecord(ctx->ev[1], ctx->st));
        if (nb) TRY(run_decode_blocks(ctx, nb, c.L, 0, c.gen_mode == 1, c.fixed_len != 0, P.n_reads, P.n_edits, &nr, &ne));
        CU(cudaEventRecord(ctx->ev[2], ctx->st));
        S.n_blocks = nb; S.n_reads = nr; S.n_edits = ne;
    }
    uint64_t n_sel = 0;
    if (nr && !iv.empty()) TRY(run_region_select(ctx, nr, iv, runs, &n_sel));
    *nr_out = nr; *ne_out = ne; *n_sel_out = n_sel; *max_len_out = max_len; *fixed_len_out = fixed_len;
    return 0;
}

extern "C" int cbcg_decode_region(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                                  const cbcg_region *regions, uint32_t n_regions,
                                  uint8_t *seq_out, uint64_t seq_cap, uint64_t *seq_len,
                                  uint64_t *read_ids, uint64_t ids_cap, uint64_t *n_reads) {
    if (!ctx || !seq_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_decode_region: bad argument");
    *seq_len = 0; if (n_reads) *n_reads = 0;
    uint64_t nr = 0, ne = 0, n_sel = 0, bytes = 0; uint32_t max_len = 1, fixed_len = 0;
    cbcg_stats &S = ctx->stats;
    TRY(region_records(ctx, in, in_len, legacy, regions, n_regions, &nr, &ne, &n_sel, &max_len, &fixed_len));
    if (n_sel) {
        TRY(run_reconstruct(ctx, n_sel, max_len, fixed_len, ctx->sel_chr.as<uint32_t>(), 0u, ctx->sel_recs.as<cbcg_read_rec>()));
        TRY(fetch_words(ctx));
        TRY(device_error(ctx, "read reconstruction"));
        cudaEventElapsedTime(&S.ms_k3, ctx->kev[2], ctx->kev[3]);
        bytes = ctx->hw->total_bytes;
    }
    CU(cudaEventRecord(ctx->ev[3], ctx->st));
    *seq_len = bytes; if (n_reads) *n_reads = n_sel;
    ctx->dec_bytes = bytes; ctx->dec_n_reads = n_sel; ctx->have_decoded = true;
    if (bytes > seq_cap || (!seq_out && bytes) || (read_ids && n_sel > ids_cap))
        return fail(ctx, CBCG_ERR_CAPACITY, "%llu reads / %llu bytes of text selected, room for %llu / %llu", (unsigned long long)n_sel,
                    (unsigned long long)bytes, (unsigned long long)ids_cap, (unsigned long long)seq_cap);
    CU(cudaEventRecord(ctx->ev[4], ctx->st));
    if (bytes) CU(cudaMemcpyAsync(seq_out, ctx->seq_out.p, bytes, cudaMemcpyDeviceToHost, ctx->st));
    if (read_ids && n_sel) CU(cudaMemcpyAsync(read_ids, ctx->sel_ids.p, n_sel * 8, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaEventRecord(ctx->ev[5], ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    cudaEventElapsedTime(&S.ms_h2d, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&S.ms_code, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&S.ms_reconstruct, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&S.ms_d2h, ctx->ev[4], ctx->ev[5]);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[5]);
    S.d2h_bytes = bytes + (read_ids ? n_sel * 8 : 0);
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ CIGAR recovery
 * (SURVEY.md 8f row 4; kernels and the meaning of the classes: k4_cigar.cu.) The side section of a batch, "CBCC":
 *   u32 magic, u32 version (1), u64 n_reads, u64 n_entries, then per read whose class is not 0, in read order:
 *   varint(read - previous listed read), u8 class, and for class 4 varint(length) + the CIGAR text.
 * A batch whose CIGARs are all what their indels imply (configs 1-4) costs the 24 header bytes. */
#define CBCC_MAGIC 0x43434243u
extern "C" uint64_t cbcg_cigar_bound(const cbcg_batch *b) {
    if (!b) return 0;
    return 24u + b->n_reads * 16u + (b->cigar_off && b->n_reads ? b->cigar_off[b->n_reads] : 0u);
}
extern "C" int cbcg_cigar_pack(cbcg_ctx *ctx, const cbcg_batch *batch, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!ctx || !batch || !out_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_cigar_pack: bad argument");
    *out_len = 0;
    TRY(cbcg_batch_upload(ctx, batch));
    const uint64_t n = ctx->db.n_reads;
    std::vector<uint8_t> cls(n);
    if (n) {
        TRY(run_extract(ctx));
        TRY(ensure(ctx, ctx->cig_cls, n + 64));
        if (launch_cigar_class(n, ctx->recs.as<cbcg_read_rec>(), ctx->edits.as<uint16_t>(), ctx->db.cigar_off, ctx->db.cigar,
                               ctx->cig_cls.as<uint8_t>(), ctx->st))
            return fail(ctx, CBCG_ERR_CUDA, "CIGAR class launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        CU(cudaMemcpyAsync(cls.data(), ctx->cig_cls.p, n, cudaMemcpyDeviceToHost, ctx->st));
        CU(cudaStreamSynchronize(ctx->st));
    }
    std::vector<uint8_t> sec(24);
    uint64_t entries = 0, prev = 0;
    for (uint64_t r = 0; r < n; r++) {
        if (!cls[r]) continue;
        put_varint(sec, r - prev); prev = r;
        sec.push_back(cls[r]);
        if (cls[r] >= 4u) {
            const uint64_t a = batch->cigar_off[r], l = batch->cigar_off[r + 1] - a;
            put_varint(sec, l);
            sec.insert(sec.end(), batch->cigar + a, batch->cigar + a + l);
        }
        entries++;
    }
    const uint32_t magic = CBCC_MAGIC, version = 1u;
    memcpy(&sec[0], &magic, 4); memcpy(&sec[4], &version, 4); memcpy(&sec[8], &n, 8); memcpy(&sec[16], &entries, 8);
    *out_len = sec.size();
    if (!out || sec.size() > out_cap) return fail(ctx, CBCG_ERR_CAPACITY, "CIGAR section is %llu bytes, room for %llu", (unsigned long long)sec.size(), (unsigned long long)out_cap);
    memcpy(out, sec.data(), sec.size());
    return CBCG_OK;
}
/* A CIGAR side section (layout above cbcg_cigar_bound) for a container of n reads -> a class per read and the class-4 texts. */
static int parse_cigar_section(cbcg_ctx *ctx, const uint8_t *section, uint64_t section_len, uint64_t n, std::vector<uint8_t> &cls,
                               std::vector<uint64_t> &exc_read, std::vector<uint64_t> &exc_off, std::vector<uint8_t> &exc_text) {
    uint32_t magic = 0, version = 0; uint64_t sn = 0, entries = 0;
    if (section_len < 24) return fail(ctx, CBCG_ERR_FORMAT, "CIGAR section too short");
    memcpy(&magic, section, 4); memcpy(&version, section + 4, 4); memcpy(&sn, section + 8, 8); memcpy(&entries, section + 16, 8);
    if (magic != CBCC_MAGIC || version != 1u) return fail(ctx, CBCG_ERR_FORMAT, "not a CIGAR section");
    if (sn != n) return fail(ctx, CBCG_ERR_FORMAT, "CIGAR section of %llu reads beside a container of %llu", (unsigned long long)sn, (unsigned long long)n);
    cls.assign(n, 0); exc_read.clear(); exc_off.assign(1, 0); exc_text.clear();
    uint64_t o = 24, prev = 0;
    for (uint64_t k = 0; k < entries; k++) {
        uint64_t d = 0, l = 0;
        if (!get_varint(section, section_len, o, d) || o >= section_len) return fail(ctx, CBCG_ERR_FORMAT, "CIGAR section truncated");
        const uint64_t r = prev + d;
        if (r >= n || (k && d == 0)) return fail(ctx, CBCG_ERR_FORMAT, "CIGAR section lists read %llu", (unsigned long long)r);
        prev = r;
        const uint8_t c = section[o++];
        if (c == 0 || c > 4) return fail(ctx, CBCG_ERR_FORMAT, "CIGAR section: class %u", (unsigned)c);
        cls[r] = c;
        if (c == 4) {
            if (!get_varint(section, section_len, o, l) || l > section_len - o) return fail(ctx, CBCG_ERR_FORMAT, "CIGAR section truncated");
            exc_read.push_back(r);
            exc_text.insert(exc_text.end(), section + o, section + o + l);
            exc_off.push_back(exc_text.size());
            o += l;
        }
    }
    return 0;
}

/* container (or legacy stream) + its section -> the CIGAR of every read, '\n'-terminated, in read order. section == NULL:
 * every read gets the CIGAR its indels imply (soft clips read as insertions). */
extern "C" int cbcg_cigar_unpack(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy, const uint8_t *section, uint64_t section_len,
                                 uint8_t *cigar_out, uint64_t cigar_cap, uint64_t *cigar_len, uint64_t *n_reads) {
    if (!ctx || !cigar_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_cigar_unpack: bad argument");
    *cigar_len = 0; if (n_reads) *n_reads = 0;
    uint64_t nr = 0, ne = 0; uint32_t max_len = 1, fixed_len = 0;
    TRY(decode_to_records(ctx, in, in_len, legacy, &nr, &ne, &max_len, &fixed_len));
    if (n_reads) *n_reads = nr;
    if (!nr) return CBCG_OK;
    std::vector<uint8_t> cls(nr, 0);
    std::vector<uint64_t> exc_read, exc_off(1, 0);
    std::vector<uint8_t> exc_text;
    uint64_t text_bound = 0;
    if (section) TRY(parse_cigar_section(ctx, section, section_len, nr, cls, exc_read, exc_off, exc_text));
    text_bound = exc_text.size() + nr * 4ull + ne * 12ull + nr * 8ull + 64;   /* per read: '\n' + <= 2 operations per indel event + 2 M runs, <= 6 bytes each */
    const uint64_t n_exc = exc_read.size();
    const uint64_t exc_bytes = (n_exc + 1) * 16 + exc_text.size() + 64;
    TRY(ensure(ctx, ctx->cig_cls, nr + 64));
    TRY(ensure(ctx, ctx->cig_exc, exc_bytes));
    TRY(ensure(ctx, ctx->cig_out, text_bound));
    TRY(ensure(ctx, ctx->tile_desc, (cigar_num_tiles(nr) + 1) * 8));
    uint64_t *d_read = ctx->cig_exc.as<uint64_t>(), *d_off = d_read + n_exc;
    uint8_t *d_text = reinterpret_cast<uint8_t *>(d_off + n_exc + 1);
    CU(cudaMemcpyAsync(ctx->cig_cls.p, cls.data(), nr, cudaMemcpyHostToDevice, ctx->st));
    if (n_exc) CU(cudaMemcpyAsync(d_read, exc_read.data(), n_exc * 8, cudaMemcpyHostToDevice, ctx->st));
    CU(cudaMemcpyAsync(d_off, exc_off.data(), (n_exc + 1) * 8, cudaMemcpyHostToDevice, ctx->st));
    if (!exc_text.empty()) CU(cudaMemcpyAsync(d_text, exc_text.data(), exc_text.size(), cudaMemcpyHostToDevice, ctx->st));
    CU(cudaMemsetAsync(wptr<unsigned long long>(ctx, W_OFF(err)), 0, 8, ctx->st));
    if (launch_cigar_emit(nr, ctx->recs.as<cbcg_read_rec>(), ctx->edits.as<uint16_t>(), ctx->cig_cls.as<uint8_t>(), d_read, d_off, d_text, n_exc,
                          ctx->cig_out.as<uint8_t>(), text_bound, ctx->tile_desc.as<uint64_t>(), wptr<uint32_t>(ctx, W_OFF(ticket)),
                          wptr<uint64_t>(ctx, W_OFF(total_bytes)), wptr<unsigned long long>(ctx, W_OFF(err)), ctx->st))
        return fail(ctx, CBCG_ERR_CUDA, "CIGAR emit launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    ctx->stats.kernel_launches++;
    TRY(fetch_words(ctx));                                   /* synchronises: the host vectors above may go */
    TRY(device_error(ctx, "CIGAR recovery"));
    const uint64_t bytes = ctx->hw->total_bytes;
    *cigar_len = bytes;
    if (bytes > cigar_cap || !cigar_out) return fail(ctx, CBCG_ERR_CAPACITY, "CIGAR text is %llu bytes, room for %llu", (unsigned long long)bytes, (unsigned long long)cigar_cap);
    CU(cudaMemcpyAsync(cigar_out, ctx->cig_out.p, bytes, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ SAM output
 * cbcg_sam_header / cbcg_decode_sam (DESIGN.md, "SAM output"; the line and the MD / NM rule: k6_sam.cu). The records come
 * from the whole-container decode or from the region decode, K3 rebuilds SEQ, K6 formats the lines next to it. The CIGAR
 * side section is parsed here into a class byte per container read and the class-4 texts; K6 looks a read up by its
 * container ordinal, which is what lets a region decode recover the CIGARs. */

/* @HD, then @SQ per name; lengths: LN per name (UINT64_MAX: unknown, not written) */
static std::string sam_header_text(const std::vector<std::string> &names, const std::vector<uint64_t> *lengths) {
    std::string h = "@HD\tVN:1.6\tSO:coordinate\n";
    for (size_t k = 0; k < names.size(); k++) {
        h += "@SQ\tSN:"; h += names[k];
        if (lengths && (*lengths)[k] != UINT64_MAX) { h += "\tLN:"; h += std::to_string((unsigned long long)(*lengths)[k]); }
        h += '\n';
    }
    return h;
}
extern "C" int cbcg_sam_header(const uint8_t *in, uint64_t in_len, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!out_len) return CBCG_ERR_ARG;
    *out_len = 0;
    Container c;
    const int rc = parse_container(in, in_len, nullptr, c);
    if (rc) return rc;
    const std::string h = sam_header_text(container_names(in, c), nullptr);
    *out_len = h.size();
    if (!out || h.size() > out_cap) return CBCG_ERR_CAPACITY;
    memcpy(out, h.data(), h.size());
    return CBCG_OK;
}

extern "C" int cbcg_decode_sam(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                               const uint8_t *section, uint64_t section_len,
                               const cbcg_region *regions, uint32_t n_regions, uint32_t flags,
                               uint8_t *out, uint64_t out_cap, uint64_t *out_len,
                               uint64_t *read_ids, uint64_t ids_cap, uint64_t *n_reads) {
    if (!ctx || !out_len || (flags & ~CBCG_SAM_HEADER) || (!regions && n_regions) || (section && !section_len))
        return fail(ctx, CBCG_ERR_ARG, "cbcg_decode_sam: bad argument");
    *out_len = 0; if (n_reads) *n_reads = 0;
    if (regions) TRY(check_regions(ctx, regions, n_regions));
    if (!ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "cbcg_set_reference has not been called");
    /* the chromosome table (legacy: the loaded reference) and the read count the section must match */
    std::vector<std::string> table = ctx->names;
    uint64_t cont_reads = 0;
    if (!legacy) {
        Container c;
        if (parse_container(in, in_len, nullptr, c)) return fail(ctx, CBCG_ERR_FORMAT, "malformed container header");
        table = container_names(in, c);
        cont_reads = c.n_reads;
    }
    std::vector<uint8_t> cls;
    std::vector<uint64_t> exc_read, exc_off(1, 0);
    std::vector<uint8_t> exc_text;
    if (section && !legacy) TRY(parse_cigar_section(ctx, section, section_len, cont_reads, cls, exc_read, exc_off, exc_text));
    /* records: every read, or the region's (with their container ordinals) */
    uint64_t nr = 0, ne = 0, n_sel = 0; uint32_t max_len = 1, fixed_len = 0;
    const cbcg_read_rec *d_recs = ctx->recs.as<cbcg_read_rec>();
    const uint32_t *d_chr = nullptr; const uint64_t *d_ids = nullptr;
    uint32_t ref_hint = 0;
    if (!regions) {
        TRY(decode_to_records(ctx, in, in_len, legacy, &nr, &ne, &max_len, &fixed_len));
        if (legacy) max_len = CBCG_MAX_READ_LEN;            /* per-read lengths are coded mod 256 (src/read_compression.c:29-33) */
        else ref_hint = ref_window_from_blocks(ctx, max_len);
        n_sel = nr;
        d_recs = ctx->recs.as<cbcg_read_rec>(); d_chr = ctx->chr_out.as<uint32_t>();
    } else {
        TRY(region_records(ctx, in, in_len, legacy, regions, n_regions, &nr, &ne, &n_sel, &max_len, &fixed_len));
        d_recs = ctx->sel_recs.as<cbcg_read_rec>(); d_chr = ctx->sel_chr.as<uint32_t>(); d_ids = ctx->sel_ids.as<uint64_t>();
    }
    if (section && legacy) TRY(parse_cigar_section(ctx, section, section_len, nr, cls, exc_read, exc_off, exc_text));   /* a legacy stream is decoded whole */
    cbcg_stats &S = ctx->stats;
    std::vector<uint64_t> lengths(table.size(), UINT64_MAX);
    for (size_t k = 0; k < table.size(); k++)
        for (size_t g = 0; g < ctx->names.size(); g++)
            if (ctx->names[g] == table[k]) { lengths[k] = ctx->h_len[g]; break; }
    const std::string head = (flags & CBCG_SAM_HEADER) ? sam_header_text(table, &lengths) : std::string();
    uint64_t rec_bytes = 0;
    if (n_sel) {
        TRY(run_reconstruct(ctx, n_sel, max_len, fixed_len, d_chr, ref_hint, d_recs));
        /* an upper bound on the lines (k6_sam.cu): per read 64 bytes of fields, the name, SEQ, 16 per edit (implied CIGAR +
           MD), and per verbatim CIGAR its text, 4 per base and 5 per deleted base (<= 255) of MD */
        size_t max_name = 0;
        std::vector<uint32_t> name_len(ctx->names.size());
        for (size_t g = 0; g < ctx->names.size(); g++) { name_len[g] = (uint32_t)ctx->names[g].size(); max_name = std::max(max_name, ctx->names[g].size()); }
        const uint64_t bound = n_sel * (64u + max_name + max_len) + 16u * ne + exc_text.size() + exc_read.size() * (4u * max_len + 5u * 255u + 8u) + 64u;
        const uint64_t n_exc = exc_read.size();
        const uint64_t aux = name_len.size() * 4 + cls.size() + (2 * n_exc + 1) * 8 + exc_text.size() + 256;
        TRY(ensure(ctx, ctx->sam_aux, aux));
        TRY(ensure(ctx, ctx->sam_out, head.size() + bound + 64));
        TRY(ensure(ctx, ctx->tile_desc, (2 * sam_num_tiles(n_sel) + 1) * 8));
        uint8_t *a = ctx->sam_aux.as<uint8_t>();
        uint64_t *d_read = reinterpret_cast<uint64_t *>(a), *d_off = d_read + n_exc;
        uint32_t *d_nl = reinterpret_cast<uint32_t *>(d_off + n_exc + 1);
        uint8_t *d_cls = reinterpret_cast<uint8_t *>(d_nl + name_len.size()), *d_text = d_cls + cls.size();
        if (n_exc) CU(cudaMemcpyAsync(d_read, exc_read.data(), n_exc * 8, cudaMemcpyHostToDevice, ctx->st));
        CU(cudaMemcpyAsync(d_off, exc_off.data(), (n_exc + 1) * 8, cudaMemcpyHostToDevice, ctx->st));
        CU(cudaMemcpyAsync(d_nl, name_len.data(), name_len.size() * 4, cudaMemcpyHostToDevice, ctx->st));
        if (!cls.empty()) CU(cudaMemcpyAsync(d_cls, cls.data(), cls.size(), cudaMemcpyHostToDevice, ctx->st));
        if (!exc_text.empty()) CU(cudaMemcpyAsync(d_text, exc_text.data(), exc_text.size(), cudaMemcpyHostToDevice, ctx->st));
        if (!head.empty()) CU(cudaMemcpyAsync(ctx->sam_out.p, head.data(), head.size(), cudaMemcpyHostToDevice, ctx->st));
        if (launch_sam(n_sel, d_recs, d_chr, ctx->edits.as<uint16_t>(), ctx->dg, ctx->g_names.as<uint8_t>(), d_nl, ctx->seq_out.as<uint8_t>(),
                       max_len, fixed_len, d_ids, section ? d_cls : nullptr, d_read, d_off, d_text, n_exc,
                       ctx->sam_out.as<uint8_t>() + head.size(), bound, ctx->tile_desc.as<uint64_t>(), wptr<uint32_t>(ctx, W_OFF(ticket)),
                       wptr<uint64_t>(ctx, W_OFF(total_bytes)), wptr<unsigned long long>(ctx, W_OFF(err)), ctx->st))
            return fail(ctx, CBCG_ERR_CUDA, "K6 launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        ctx->stats.kernel_launches++;
        CU(cudaEventRecord(ctx->ev[3], ctx->st));
        TRY(fetch_words(ctx));                               /* synchronises: the host vectors above may go */
        TRY(device_error(ctx, "SAM output"));
        cudaEventElapsedTime(&S.ms_k3, ctx->kev[2], ctx->kev[3]);
        rec_bytes = ctx->hw->total_bytes;
    } else {
        TRY(ensure(ctx, ctx->sam_out, head.size() + 64));
        if (!head.empty()) CU(cudaMemcpyAsync(ctx->sam_out.p, head.data(), head.size(), cudaMemcpyHostToDevice, ctx->st));
        CU(cudaEventRecord(ctx->ev[3], ctx->st));
    }
    /* the SAM text becomes "the decoded text" that cbcg_fetch_decoded returns */
    std::swap(ctx->seq_out, ctx->sam_out);
    const uint64_t bytes = head.size() + rec_bytes;
    *out_len = bytes; if (n_reads) *n_reads = n_sel;
    ctx->dec_bytes = bytes; ctx->dec_n_reads = n_sel; ctx->have_decoded = true;
    if (bytes > out_cap || (!out && bytes) || (read_ids && n_sel > ids_cap))
        return fail(ctx, CBCG_ERR_CAPACITY, "%llu reads / %llu bytes of SAM, room for %llu / %llu", (unsigned long long)n_sel,
                    (unsigned long long)bytes, (unsigned long long)ids_cap, (unsigned long long)out_cap);
    CU(cudaEventRecord(ctx->ev[4], ctx->st));
    if (bytes) CU(cudaMemcpyAsync(out, ctx->seq_out.p, bytes, cudaMemcpyDeviceToHost, ctx->st));
    if (read_ids && n_sel) {
        if (d_ids) CU(cudaMemcpyAsync(read_ids, d_ids, n_sel * 8, cudaMemcpyDeviceToHost, ctx->st));
        else for (uint64_t r = 0; r < n_sel; r++) read_ids[r] = r;
    }
    CU(cudaEventRecord(ctx->ev[5], ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    cudaEventElapsedTime(&S.ms_h2d, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&S.ms_code, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&S.ms_reconstruct, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&S.ms_d2h, ctx->ev[4], ctx->ev[5]);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[5]);
    S.d2h_bytes = bytes + (read_ids && d_ids ? n_sel * 8 : 0);
    return CBCG_OK;
}

/* K2d + K3 on the blocks of the last cbcg_encode_resident, everything staying in HBM. */
extern "C" int cbcg_decode_resident(cbcg_ctx *ctx) {
    if (!ctx) return CBCG_ERR_ARG;
    if (!ctx->have_encoded) return fail(ctx, CBCG_ERR_ARG, "nothing encoded yet");
    CU(cudaSetDevice(ctx->device));
    set_carveout_all(-1);
    ctx->have_decoded = false;
    cbcg_stats &S = ctx->stats;
    S.ms_code = S.ms_reconstruct = S.ms_plan = S.ms_total = S.ms_extract = S.ms_gather = 0; S.kernel_launches = 0;
    const uint64_t nb = ctx->enc_n_blocks;
    if (!nb) { ctx->dec_bytes = 0; ctx->dec_n_reads = 0; ctx->have_decoded = true; return CBCG_OK; }
    const int legacy = (int)ctx->enc_legacy;
    ctx->layout_mode = ctx->enc_layout_mode;
    /* hblocks still hold the encoder's descriptors (n_reads, chr, base_pos, n_edits, payload_bytes); the compact
       payload is in ctx->payload in block order. */
    uint64_t nr = 0, ne = 0;
    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    if (legacy) { ctx->hblocks[0].n_reads = (uint32_t)ctx->enc_n_reads + 1u; ctx->hblocks[0].n_edits = (uint32_t)ctx->enc_n_edits + 64u; }
    gens_from_blocks(ctx, nb);
    TRY(run_decode_blocks(ctx, nb, legacy ? 0u : ctx->enc_L, legacy, !legacy && ctx->enc_gen_mode == 1, !legacy && ctx->enc_fixed,
                          legacy ? ctx->enc_n_reads + 1u : ctx->enc_n_reads,
                          legacy ? ctx->enc_n_edits + 64u : ctx->enc_n_edits, &nr, &ne));
    CU(cudaEventRecord(ctx->ev[1], ctx->st));
    if (nr) {
        TRY(run_reconstruct(ctx, nr, legacy ? CBCG_MAX_READ_LEN : std::max(ctx->enc_max_len, 1u),
                            (!legacy && ctx->enc_fixed) ? ctx->enc_L : 0u, ctx->chr_out.as<uint32_t>(),
                            legacy ? 0u : ref_window_from_blocks(ctx, std::max(ctx->enc_max_len, 1u))));
        CU(cudaEventRecord(ctx->ev[2], ctx->st));
        TRY(fetch_words(ctx));
        TRY(device_error(ctx, "read reconstruction"));
        cudaEventElapsedTime(&S.ms_k3, ctx->kev[2], ctx->kev[3]);
        ctx->dec_bytes = ctx->hw->total_bytes;
    } else { CU(cudaEventRecord(ctx->ev[2], ctx->st)); CU(cudaStreamSynchronize(ctx->st)); ctx->dec_bytes = 0; }
    ctx->dec_n_reads = nr; ctx->have_decoded = true;
    cudaEventElapsedTime(&S.ms_code, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&S.ms_reconstruct, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[2]);
    S.n_reads = nr; S.n_edits = ne; S.n_blocks = nb;
    if (legacy) { ctx->hblocks[0].n_reads = (uint32_t)ctx->enc_n_reads; ctx->hblocks[0].n_edits = (uint32_t)ctx->enc_n_edits; }
    return CBCG_OK;
}

extern "C" int cbcg_fetch_decoded(cbcg_ctx *ctx, uint8_t *seq_out, uint64_t seq_cap, uint64_t *seq_len) {
    if (!ctx || !seq_len) return fail(ctx, CBCG_ERR_ARG, "cbcg_fetch_decoded: bad argument");
    if (!ctx->have_decoded) return fail(ctx, CBCG_ERR_ARG, "nothing decoded yet");
    *seq_len = ctx->dec_bytes;
    if (ctx->dec_bytes > seq_cap || (!seq_out && ctx->dec_bytes)) return fail(ctx, CBCG_ERR_CAPACITY, "decoded text is %llu bytes", (unsigned long long)ctx->dec_bytes);
    CU(cudaSetDevice(ctx->device));
    if (ctx->dec_bytes) CU(cudaMemcpyAsync(seq_out, ctx->seq_out.p, ctx->dec_bytes, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    return CBCG_OK;
}

/* ------------------------------------------------------------------------------------------------ K3 alone */
extern "C" int cbcg_reconstruct(cbcg_ctx *ctx, uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr,
                                const uint16_t *edits, uint64_t n_edits, uint8_t *seq_out, uint64_t seq_cap,
                                uint64_t *seq_len) {
    if (!ctx || !seq_len || (n_reads && (!recs || !chr)) || (n_edits && !edits)) return fail(ctx, CBCG_ERR_ARG, "cbcg_reconstruct: bad argument");
    if (!ctx->dg.n_chr) return fail(ctx, CBCG_ERR_NO_REFERENCE, "cbcg_set_reference has not been called");
    CU(cudaSetDevice(ctx->device));
    *seq_len = 0;
    ctx->stats = cbcg_stats();
    if (!n_reads) return CBCG_OK;
    uint32_t max_len = 1, min_len = 0xffffffffu;
    for (uint64_t r = 0; r < n_reads; r++) {
        if (recs[r].len > max_len) max_len = recs[r].len;
        if (recs[r].len < min_len) min_len = recs[r].len;
        if (!recs[r].match && (uint64_t)recs[r].edit_off + recs[r].n_dels + recs[r].n_snps + recs[r].n_ins > n_edits)
            return fail(ctx, CBCG_ERR_ARG, "read %llu: edit range outside the edit array", (unsigned long long)r);
    }
    if (max_len > CBCG_MAX_READ_LEN) return fail(ctx, CBCG_ERR_INPUT, "read longer than %u", CBCG_MAX_READ_LEN);
    TRY(ensure(ctx, ctx->recs, (n_reads + 1) * sizeof(cbcg_read_rec)));
    TRY(ensure(ctx, ctx->chr_out, (n_reads + 1) * 4));
    TRY(ensure(ctx, ctx->edits, (n_edits + 64) * 2));
    CU(cudaMemcpyAsync(ctx->recs.p, recs, n_reads * sizeof(cbcg_read_rec), cudaMemcpyHostToDevice, ctx->st));
    CU(cudaMemcpyAsync(ctx->chr_out.p, chr, n_reads * 4, cudaMemcpyHostToDevice, ctx->st));
    if (n_edits) CU(cudaMemcpyAsync(ctx->edits.p, edits, n_edits * 2, cudaMemcpyHostToDevice, ctx->st));
    TRY(reset_words(ctx));
    CU(cudaEventRecord(ctx->ev[0], ctx->st));
    TRY(run_reconstruct(ctx, n_reads, max_len, min_len == max_len ? max_len : 0u, ctx->chr_out.as<uint32_t>()));
    CU(cudaEventRecord(ctx->ev[1], ctx->st));
    TRY(fetch_words(ctx));
    cudaEventElapsedTime(&ctx->stats.ms_reconstruct, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->stats.ms_k3, ctx->kev[2], ctx->kev[3]);
    TRY(device_error(ctx, "read reconstruction"));
    const uint64_t bytes = ctx->hw->total_bytes;
    *seq_len = bytes;
    ctx->dec_bytes = bytes; ctx->dec_n_reads = n_reads; ctx->have_decoded = true;
    if (bytes > seq_cap || !seq_out) return fail(ctx, CBCG_ERR_CAPACITY, "text is %llu bytes, room for %llu", (unsigned long long)bytes, (unsigned long long)seq_cap);
    CU(cudaMemcpyAsync(seq_out, ctx->seq_out.p, bytes, cudaMemcpyDeviceToHost, ctx->st));
    CU(cudaStreamSynchronize(ctx->st));
    ctx->stats.n_reads = n_reads; ctx->stats.n_edits = n_edits;
    return CBCG_OK;
}
