// rt_deflate.cuh -- the deflate pieces that the PNG (rt_png.cu) and OpenEXR (rt_exr.cu) encoders share: fixed-Huffman
// literal and length codes, the framing of a byte-aligned piece, and the Adler-32 modulus.
//
// A piece is a non-final fixed-Huffman block (3-bit header, the tokens, end-of-block) followed by an empty non-final
// stored block, so it starts and ends on a byte and decodes without its neighbours; a zlib stream is "78 01", pieces
// back to back, "03 00" (a final empty fixed block) and the Adler-32 of the data.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace {

constexpr uint32_t ADLER_MOD = 65521u;
constexpr uint32_t FULL = 0xffffffffu;

__constant__ uint16_t c_len_base[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23, 27,
                                        31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};

// ---- fixed Huffman codes (RFC 1951 3.2.6), bit-reversed for the LSB-first stream --------------------------------
__device__ __forceinline__ uint32_t lit_bits(uint32_t v) { return v < 144u ? 8u : 9u; }

__device__ __forceinline__ uint32_t lit_code(uint32_t v) {
    return v < 144u ? __brev(0x30u + v) >> 24 : __brev(0x190u + v - 144u) >> 23;
}

// length L (3..258) + a distance whose code and extra bits are `dist` (dist_bits long, LSB-first): one token of at
// most 8 + 5 + dist_bits bits
__device__ __forceinline__ uint32_t match_code(uint32_t L, uint32_t dist, uint32_t dist_bits, uint32_t *bits) {
    int k = 28;
    while (c_len_base[k] > L) k--;
    const uint32_t sym = 257u + (uint32_t)k;
    uint32_t c, n;
    if (sym < 280u) c = __brev(sym - 256u) >> 25, n = 7;
    else c = __brev(0xC0u + sym - 280u) >> 24, n = 8;
    c |= (L - c_len_base[k]) << n;
    n += c_len_extra[k];
    c |= dist << n;
    *bits = n + dist_bits;
    return c;
}

// Bytes of a piece: the staged token bits, zeros (end-of-block, the stored block's header, padding), then the stored
// block's LEN / NLEN 00 00 FF FF.
__device__ __forceinline__ uint32_t piece_bytes(uint32_t bits) { return (bits + 10u + 7u) / 8u + 4u; }

__device__ __forceinline__ uint32_t piece_byte(const uint8_t *staged, uint32_t bits, uint32_t len, uint32_t q) {
    return q < (bits + 7u) / 8u ? staged[q] : (q + 2u >= len ? 0xffu : 0u);
}

}  // namespace
