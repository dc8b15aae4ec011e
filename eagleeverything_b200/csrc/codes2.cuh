// 2-bit genotype codes <-> int8 store bytes, shared by the packed container (pack2.cu) and the PLINK .bed decoder (bed.cu).
// A 32-bit word holds 16 codes, genotype k in bits 2k, 2k+1 (the order of both formats); codes are those of the ASCII
// file (0 = AA, 1 = AB / missing, 2 = BB) and a store byte is 1 - code (decode.cu explains the sign).
#pragma once
#include <cstdint>

namespace eg {

// address of genotype (r, c) of a store: row-major (pitch > 0) or K-blocked [c/128][rows][128] (pitch == 0)
__device__ __forceinline__ int64_t store_off(int64_t r, int64_t c, int64_t rows, int64_t pitch) {
    return pitch ? r * pitch + c : ((c >> 7) * rows + r) * 128 + (c & 127);
}

// 16 store bytes (1 - code) -> 32 bits of 2-bit codes
__device__ __forceinline__ uint32_t pack16(uint4 v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t out = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        // store byte +1 / 0 / -1 (= 1 - code, decode.cu) -> code 0 / 1 / 2: bit 1 = sign, bit 0 = !(low bit)
        const uint32_t c = ((w[k] >> 6) & 0x02020202u) | (~w[k] & 0x01010101u);
        const uint32_t p = (c | (c >> 6) | (c >> 12) | (c >> 18)) & 0xFFu;  // the four 2-bit codes into one byte
        out |= p << (8 * k);
    }
    return out;
}
// 32 bits of 2-bit codes -> 16 int8 genotypes; bad |= 1 when a code is 3
__device__ __forceinline__ uint4 unpack16(uint32_t bits, uint32_t& bad) {
    bad |= (bits & (bits >> 1) & 0x55555555u) ? 1u : 0u;
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t b = (bits >> (8 * k)) & 0xFFu;
        const uint32_t c = (b & 3u) | ((b & 0xCu) << 6) | ((b & 0x30u) << 12) | ((b & 0xC0u) << 18);  // one code per byte
        w[k] = (0x81818181u - c) ^ 0x80808080u;                                                     // bytewise 1 - code
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

}  // namespace eg
