/*
 * k2_blocks.cu -- K2 for blocked containers, the one-thread-per-block kernels built on the scalar coder of
 * k2_roles.cuh (K2Ac): the interval half of a two-kernel encode, and the initial generation snapshot.
 *
 * The interval kernel is latency-bound integer work with a few hundred warps in flight: one warp per CTA lets the
 * hardware spread them over all SMs (one warp per scheduler runs its dependent chain at the full issue rate).
 */
#include "common.cuh"
#include "k2_roles.cuh"

#define K2R_LANES 32u

/* ------------------------------------------------------------------------------------------------
 * The interval half of a two-kernel encode (k2_coder.cu, k2_model_kernel): ONE THREAD PER BLOCK walks the block's
 * intervals in stream order through the arithmetic coder (arithmetic_encoder_step, src/Arithmetic_stream.c:274-345,
 * closed form: ac_core.h) and the MSB-first bit packer (:155-194). A warp holds 32 consecutive blocks. With one warp
 * per SM nothing hides a dependent instruction's latency, so the time of a block is the length of the dependent chain
 * per symbol: the step is written WITHOUT BRANCHES (selects and predicated stores) and four symbols at a time, so that
 * the compiler overlaps what hangs off the interval (bit packing, the next symbols' reciprocals and conversions) with
 * the chain through it (range -> two quotients -> shared-prefix shift -> E3 shift). What the straight-line step does not
 * cover -- a POS escape (its four byte symbols come from the escape list), an E3 run that does not fit one 32-bit put,
 * a full payload region -- raises a flag; the group of four is then redone from the saved state by the general coder. */
struct K2CState { uint32_t l, u, scale3, nacc, out_pos; uint64_t acc; };
/* Four symbols in three passes, so that the order of the instructions is the order of their dependences (one warp per SM
 * issues in order: whatever stands between two links of the chain through the interval delays it):
 *   1. what depends on the slots alone: the reciprocal of the total, the bounds as doubles;
 *   2. the chain: range -> two quotients (ac_muldiv's estimate and remainder fix) -> shared-prefix shift -> E3 shift;
 *   3. the bits: packing and the predicated store, a short chain of its own through the accumulator. */
__device__ __forceinline__ uint32_t k2c_fast4(K2CState &s, const uint4 (&t)[4], uint8_t *out, uint32_t out_cap) {
    /* pass 1 turns each bound into a 32-bit fraction of the total, F = trunc(bound * 2^32 / n) (within one of the floor:
       the reciprocal is good to 2^-44; a bound equal to the total saturates to 2^32 - 1), so that the chain's quotient
       floor(range * bound / n) is ONE integer multiply-high, off by at most one like ac_muldiv's estimate and put right by
       the same remainder test -- the FP64 conversions and multiplies (the longest latencies of the step) leave the chain. */
    uint32_t fh[4], fl[4], hi[4], slow = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        hi[q] = t[q].x + t[q].y;
        const double r32 = __dmul_rn(ac_rcp(t[q].z), 4294967296.0);
        fh[q] = __double2uint_rz(__dmul_rn(__uint2double_rn(hi[q]), r32));
        fl[q] = __double2uint_rz(__dmul_rn(__uint2double_rn(t[q].x), r32));
        slow |= (t[q].w != 0u) | (t[q].y == 0u) | (t[q].z == 0u);
    }
    uint32_t k[4], bits[4], m[4];
    uint32_t l = s.l, u = s.u;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint32_t range = u - l + 1u, n = t[q].z;
        uint32_t qh = __umulhi(range, fh[q]), ql = __umulhi(range, fl[q]);
        const int32_t rh = (int32_t)(range * hi[q] - qh * n), rl = (int32_t)(range * t[q].x - ql * n);   /* estimates are off by at most one */
        qh += rh < 0 ? 0xffffffffu : (rh >= (int32_t)n ? 1u : 0u);
        ql += rl < 0 ? 0xffffffffu : (rl >= (int32_t)n ? 1u : 0u);
        AcInterval a = { l + ql, l + qh - 1u }, nx;
        ac_renorm_shape(a, k[q], bits[q], m[q], nx);
        l = nx.l; u = nx.u;
    }
    s.l = l; s.u = u;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        /* the k shared bits: the first, then the pending E3 bits inverted (:318-322), then the other k - 1 */
        const uint32_t run = k[q] ? s.scale3 : 0u;
        const uint32_t nb = k[q] ? k[q] + run : 0u;
        const uint32_t rest_bits = k[q] ? k[q] - 1u : 0u;
        const uint32_t b0 = (bits[q] >> rest_bits) & 1u;
        const uint32_t inv = b0 ? 0u : 0xffffffffu;
        const uint32_t runc = run & 31u, sh = (runc + rest_bits) & 31u;      /* in range whenever nb <= 32 */
        const uint32_t v = (b0 << sh) | ((inv & ((1u << runc) - 1u)) << rest_bits) | (bits[q] & ((1u << rest_bits) - 1u));
        slow |= (nb > 32u);
        const uint64_t acc = (s.acc << (nb & 63u)) | (uint64_t)v;           /* bits above nacc are never read: no masking */
        const uint32_t nacc = s.nacc + nb;
        const bool full = nacc >= 32u;
        const bool room = s.out_pos + 4u <= out_cap;
        slow |= (uint32_t)(full && !room);
        if (full && room) *reinterpret_cast<uint32_t *>(out + s.out_pos) = __byte_perm((uint32_t)(acc >> ((nacc - 32u) & 63u)), 0u, 0x0123);
        s.out_pos += full ? 4u : 0u;
        s.nacc = full ? nacc - 32u : nacc;
        s.acc = acc;
        s.scale3 = (k[q] ? 0u : s.scale3) + m[q];
    }
    return slow;
}
/* the general coder over `count` main slots from T (and the escapes they flag) */
__device__ __noinline__ int k2c_general(K2CState *st, const uint4 *T, uint32_t count, const uint4 **escp, uint8_t *out, uint32_t out_cap, uint32_t *nsym) {
    K2Ac ac;
    ac.init_enc(out, out_cap);
    ac.a.l = st->l; ac.a.u = st->u; ac.scale3 = (int32_t)st->scale3; ac.acc = st->acc; ac.nacc = st->nacc; ac.out_pos = st->out_pos;
    const uint4 *esc = *escp;
    for (uint32_t i = 0; i < count; i++) {
        const uint4 t = T[i];
        ac.encode(t.x, t.y, t.z);
        if (t.w) {                                           /* POS escape: its four byte symbols (compress_pos_alpha :75-108) */
            for (uint32_t k = 0; k < 4u; k++) ac.encode(esc[k].x, esc[k].y, esc[k].z);
            esc += 4;
        }
    }
    *escp = esc;
    st->l = ac.a.l; st->u = ac.a.u; st->scale3 = (uint32_t)ac.scale3; st->acc = ac.acc; st->nacc = ac.nacc; st->out_pos = ac.out_pos;
    *nsym += ac.nsym;
    return ac.err;
}
#define K2C_GROUP 4u
__global__ void __launch_bounds__(K2R_LANES)
k2_code_kernel(CoderParams P) {
    if (*reinterpret_cast<volatile unsigned long long *>(P.err)) return;    /* an earlier stage failed: slots may be unwritten */
    const uint32_t bl = blockIdx.x * K2R_LANES + threadIdx.x;
    if (bl >= P.n_blocks) return;
    const uint32_t b = P.block_begin + bl;
    BlockDesc &B = P.blocks[b];
    const uint4 *T = reinterpret_cast<const uint4 *>(P.tri) + k2_tri_off(B, b);
    const uint32_t total = T[0].x;
    const uint4 *esc = T + k2_tri_esc(B);
    const uint4 *src = T + 1;
    uint8_t *out = P.payload + B.payload_off;
    const uint32_t out_cap = (uint32_t)payload_cap_bytes(B.n_reads, B.n_edits, 1);
    K2CState st = { 0u, CBCG_AC_TOP, 0u, 0u, 0u, 0ull };
    uint32_t nsym = 0; int err = 0;
    const uint32_t groups = total / K2C_GROUP;
    uint4 nxt[K2C_GROUP];
#pragma unroll
    for (uint32_t q = 0; q < K2C_GROUP; q++) nxt[q] = groups ? src[q] : make_uint4(0u, 1u, 1u, 0u);
    for (uint32_t g = 0; g < groups && !err; g++) {
        uint4 cur[K2C_GROUP];
#pragma unroll
        for (uint32_t q = 0; q < K2C_GROUP; q++) cur[q] = nxt[q];
        if (g + 1u < groups) {
#pragma unroll
            for (uint32_t q = 0; q < K2C_GROUP; q++) nxt[q] = src[(g + 1u) * K2C_GROUP + q];
        }
        /* the loads above are a group ahead of their use, which does not cover a miss to HBM (13 % of the stall samples
           waited for them): ask for the line four groups ahead */
        if (g + 4u < groups) asm volatile("prefetch.global.L1 [%0];" ::"l"(src + (g + 4u) * K2C_GROUP));
        const K2CState saved = st;
        uint32_t slow = 0;
        slow = k2c_fast4(st, cur, out, out_cap);
        if (K2R_UNLIKELY(slow)) {                            /* through copies: the state itself stays in registers */
            K2CState tmp = saved; const uint4 *e2 = esc; uint32_t ns2 = 0;
            err = k2c_general(&tmp, src + g * K2C_GROUP, K2C_GROUP, &e2, out, out_cap, &ns2);
            st = tmp; esc = e2; nsym += ns2;
        } else nsym += K2C_GROUP;
    }
    if (!err && (total % K2C_GROUP)) {
        K2CState tmp = st; const uint4 *e2 = esc; uint32_t ns2 = 0;
        err = k2c_general(&tmp, src + groups * K2C_GROUP, total % K2C_GROUP, &e2, out, out_cap, &ns2);
        st = tmp; nsym += ns2;
    }
    if (!err) {                                              /* 1 + pending bits, zeros ever after (K2Ac::finish_short) */
        K2Ac ac;
        ac.init_enc(out, out_cap);
        ac.a.l = st.l; ac.a.u = st.u; ac.scale3 = (int32_t)st.scale3; ac.acc = st.acc; ac.nacc = st.nacc; ac.out_pos = st.out_pos; ac.nsym = nsym;
        ac.finish_short();
        err = ac.err; st.out_pos = ac.out_pos;
    }
    if (err) { dev_set_error(P.err, err, (uint64_t)b << 20); return; }
    B.n_symbols = nsym; B.payload_bytes = st.out_pos; B.sub_bytes[0] = st.out_pos;
}
int launch_code_kernel(const CoderParams &p, cudaStream_t st) {
    if (p.n_blocks == 0) return 0;
    k2_code_kernel<<<(p.n_blocks + K2R_LANES - 1u) / K2R_LANES, K2R_LANES, 0, st>>>(p);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

__global__ void __launch_bounds__(32) k2_snapshot_init_kernel(uint8_t *snap, uint32_t L) {
    if (threadIdx.x == 0) k2_snapshot_init(snap, L);
}
int launch_snapshot_init(uint8_t *snap, uint32_t L, cudaStream_t st) {
    k2_snapshot_init_kernel<<<1, 32, 0, st>>>(snap, L);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
void blocks_set_carveout(int pct) {
    cudaFuncSetAttribute(k2_snapshot_init_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k2_code_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
}
