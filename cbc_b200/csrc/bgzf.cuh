/* bgzf.cuh -- CRC32 of gzip / BGZF members (SAMv1 4.1), shared by K9 (BGZF output) and K10 (BGZF input): the byte table and
 * zlib's GF(2) shift, which combines the raw CRCs of chunks that threads computed apart. */
#pragma once
#include <stdint.h>

#define BGZF_CRC_POLY 0xedb88320u

/* x^(2^k) mod P, reflected (zlib's x2n_table) */
static __constant__ uint32_t bgzf_x2n[32] = {
    0x40000000u, 0x20000000u, 0x08000000u, 0x00800000u, 0x00008000u, 0xedb88320u, 0xb1e6b092u, 0xa06a2517u, 0xed627daeu, 0x88d14467u,
    0xd7bbfe6au, 0xec447f11u, 0x8e7ea170u, 0x6427800eu, 0x4d47bae0u, 0x09fe548fu, 0x83852d0fu, 0x30362f1au, 0x7b5a9cc3u, 0x31fec169u,
    0x9fec022au, 0x6c8dedc4u, 0x15d6874du, 0x5fde7a4eu, 0xbad90e37u, 0x2e4e5eefu, 0x4eaba214u, 0xa8a472c0u, 0x429a969eu, 0x148d302au,
    0xc40ba6d0u, 0xc4e22c3cu };

/* entry k of the byte-at-a-time table: crc = tab[(crc ^ byte) & 0xff] ^ (crc >> 8) */
__device__ __forceinline__ uint32_t bgzf_crc_table_entry(uint32_t k) {
    uint32_t c = k;
    for (int j = 0; j < 8; j++) c = (c & 1u) ? (c >> 1) ^ BGZF_CRC_POLY : c >> 1;
    return c;
}

/* a * b mod P, reflected (zlib's multmodp) */
__device__ __forceinline__ uint32_t bgzf_multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (uint32_t m = 1u << 31; m; m >>= 1) {
        if (a & m) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ BGZF_CRC_POLY : b >> 1;
    }
    return p;
}
/* crc * x^(8 n) mod P: a raw CRC followed by n more bytes of zeros */
__device__ __forceinline__ uint32_t bgzf_crc_shift(uint32_t crc, uint32_t n) {
    uint32_t op = 1u << 31, k = 3;
    for (; n; n >>= 1, k++) if (n & 1u) op = bgzf_multmodp(bgzf_x2n[k & 31u], op);
    return bgzf_multmodp(op, crc);
}
/* The CRC32 of B bytes from the XOR of its chunks' raw CRCs, each shifted past the bytes after its chunk (raw: initial value
   0, no final inversion): the initial value's contribution shifted past the whole, then the final inversion. */
__device__ __forceinline__ uint32_t bgzf_crc_finish(uint32_t raw_all, uint32_t B) {
    return raw_all ^ bgzf_crc_shift(0xffffffffu, B) ^ 0xffffffffu;
}
