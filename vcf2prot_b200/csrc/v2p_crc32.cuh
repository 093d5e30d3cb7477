// v2p_crc32.cuh -- CRC-32 (gzip / BGZF, reflected polynomial 0xEDB88320) on the device: slicing-by-4 tables and the
// GF(2) algebra that moves a piece's CRC past the bytes that follow it, so that independent pieces combine:
//   crc(A || B) = gf_mul(x_pow_8n(|B|), crc(A)) ^ crc(B).
// Used by the gzip writer (v2p_gzip.cu) and the BGZF reader (v2p_inflate.cuh).  The tables are per translation unit:
// each one that includes this header launches k_crc32_init once (<<<1, 256>>>) before it uses them.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace {

constexpr uint32_t POLY = 0xEDB88320u;

__device__ uint32_t g_crc_tab[4][256];  // slicing-by-4: [k][b] = CRC of byte b followed by k zero bytes
__device__ uint32_t g_xp8[40];   // x^(8 * 2^j) mod P, reflected
__device__ uint32_t g_x64[256];  // x^(8 * 64 * k): a CRC moved past k whole pieces
__device__ uint32_t g_xb[65];    // x^(8 * m),  m = 0..64

// a*b mod P, reflected representation (bit 31 is x^0)
__device__ __forceinline__ uint32_t gf_mul(uint32_t a, uint32_t b) {
    uint32_t p = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        p ^= (a & (0x80000000u >> i)) ? b : 0u;
        b = (b >> 1) ^ ((b & 1u) ? POLY : 0u);
    }
    return p;
}

__device__ __forceinline__ uint32_t x_pow_8n(uint64_t n) {  // x^(8n) mod P
    uint32_t r = 0x80000000u;
    for (int j = 0; n; ++j, n >>= 1)
        if (n & 1) r = gf_mul(r, g_xp8[j]);
    return r;
}

__global__ void k_crc32_init() {
    const int t = threadIdx.x;
    uint32_t c = (uint32_t)t;
    for (int k = 0; k < 8; ++k) c = (c >> 1) ^ ((c & 1u) ? POLY : 0u);
    g_crc_tab[0][t] = c;
    __syncthreads();
    for (int k = 1; k < 4; ++k) {
        c = (c >> 8) ^ g_crc_tab[0][c & 255u];
        g_crc_tab[k][t] = c;
    }
    uint32_t x8 = 0x80000000u >> 8, xb = 0x80000000u, x64;  // x^8, then x^(8t) by t multiplications
    for (int k = 0; k < t && k < 65; ++k) xb = gf_mul(xb, x8);
    if (t < 65) g_xb[t] = xb;
    x64 = x8;
    for (int k = 0; k < 6; ++k) x64 = gf_mul(x64, x64);  // x^(8*64)
    uint32_t v = 0x80000000u;
    for (int k = 0; k < t; ++k) v = gf_mul(v, x64);
    g_x64[t] = v;
    if (t == 0) {
        uint32_t sq = x8;
        for (int j = 0; j < 40; ++j) {
            g_xp8[j] = sq;
            sq = gf_mul(sq, sq);
        }
    }
}

}  // namespace
