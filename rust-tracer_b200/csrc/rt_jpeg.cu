// rt_jpeg.cu -- JPEG files encoded on the device (rt_encode_jpeg, rt_render_sweep_jpeg).
//
// The layout is fixed so that there is exactly one byte string per image and quality: baseline sequential, 4:2:0, the
// standard Huffman tables of ITU T.81 Annex K, one restart interval per MCU row (16 image rows), the markers in the
// order libjpeg writes them.  The arithmetic is libjpeg's integer arithmetic throughout, so the file is the one
// libjpeg-turbo writes for the same pixels (tests/_jpeg_ref.py is the reference encoder; DESIGN.md "JPEG output").
//
// Three launches:
//   jpeg_transform   one warp per MCU: 16x16 RGBA pixels (16-byte loads), colour conversion, 2x2 chroma
//                    downsampling, the islow FDCT and quantisation of its six blocks in shared memory; the zig-zagged
//                    int16 coefficients to global memory and each block's AC bit length, from the nonzero mask by
//                    warp ballots (no serial walk).
//   jpeg_encode_rows one CTA per MCU row (one restart interval): each block's DC difference from its neighbour's DC,
//                    a scan of the block bit lengths for every block's bit offset, then one warp per block writes its
//                    codes MSB-first into the row's staging slot (a warp scan places each coefficient's codes; atomic
//                    OR, since only words at block edges are shared); the 1-bit padding and the count of 0xFF bytes.
//   jpeg_assemble    one CTA per MCU row: its place in the file from the stuffed sizes of the rows before it, the
//                    copy of its bytes with a 0x00 after every 0xFF, its RST marker; CTA 0 also writes the header,
//                    the last CTA EOI and the length word.
#include "rt_jpeg.h"

#include <string.h>

namespace {

constexpr uint32_t FULL = 0xffffffffu;
constexpr uint32_t HEADER_BYTES = 2 + 18 + 2 * 69 + 19 + 2 * 33 + 2 * 183 + 6 + 14;  // SOI .. SOS
constexpr uint32_t BLOCK_BITS = 11 + 11 + 63 * (16 + 10);  // the most one block codes to (DESIGN.md "JPEG output")
constexpr uint32_t T_WARPS = 8;     // jpeg_transform: MCUs per CTA
constexpr uint32_t E_THREADS = 1024;  // jpeg_encode_rows
constexpr uint32_t A_THREADS = 256;   // jpeg_assemble

// ITU T.81 Annex K tables: quantisation (natural order), Huffman BITS and HUFFVAL (DC luma, AC luma, DC chroma,
// AC chroma)
const uint8_t k_base_quant[2][64] = {
    {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,  14, 13, 16, 24, 40,  57,
     69, 56, 14, 17, 22,  29,  51,  87,  80, 62, 18, 22, 37,  56,  68,  109, 103, 77, 24, 35, 55, 64,
     81, 104, 113, 92, 49, 64, 78, 87,  103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99},
    {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99,
     99, 99, 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99}};
const uint8_t k_bits[4][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
                               {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
                               {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0},
                               {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
const uint8_t k_dc_vals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
const uint8_t k_ac_vals[2][162] = {
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
     0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
     0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
     0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
     0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
     0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
     0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
     0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
     0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
     0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
     0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
     0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
     0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
     0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
     0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
     0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
     0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};
// zig-zag position -> natural index
__constant__ uint8_t c_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                     12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                     35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                     58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
const uint8_t k_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                              41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                              30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// What the kernels need of a quality: the quantisation divisors 8 * qtbl (natural order; luma, chroma) and every
// Huffman code as size << 16 | code (DC luma, DC chroma; AC luma, AC chroma; unused symbols 0).
struct Tables {
    uint32_t dc[2][12];
    uint32_t ac[2][256];
    uint16_t div[2][64];
};

struct Header {  // the bytes before the first entropy-coded segment
    uint8_t b[(HEADER_BYTES + 3) / 4 * 4];
};

struct Scratch {
    int16_t *coef;     // per block: 64 quantised coefficients, zig-zag order
    uint32_t *acbits;  // per block: bits of its AC codes (with EOB)
    uint32_t *boff;    // per block: its first bit within its row's segment
    uint32_t *stage;   // per MCU row: slot_words words of the segment, MSB first
    uint2 *rows;       // per MCU row: {segment bytes with padding, 0xFF bytes among them}
    uint32_t slot_words;
};

struct Layout {
    uint32_t mcus, rows, slot_words;  // MCUs per row, MCU rows, staging words per row
    size_t blocks, coef_bytes, acbits_bytes, boff_bytes, stage_bytes, rows_bytes;
};

size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

Layout layout_of(uint32_t width, uint32_t height) {
    Layout l;
    l.mcus = (width + 15) / 16;
    l.rows = (height + 15) / 16;
    l.blocks = (size_t)l.mcus * l.rows * 6;
    l.slot_words = (uint32_t)round_up(((uint64_t)l.mcus * 6 * BLOCK_BITS + 8 + 31) / 32, 32);
    l.coef_bytes = round_up(l.blocks * 64 * sizeof(int16_t), 128);
    l.acbits_bytes = round_up(l.blocks * 4, 128);
    l.boff_bytes = round_up(l.blocks * 4, 128);
    l.stage_bytes = (size_t)l.rows * l.slot_words * 4;
    l.rows_bytes = round_up((size_t)l.rows * sizeof(uint2), 128);
    return l;
}

__device__ __forceinline__ uint32_t nbits(uint32_t a) { return 32u - __clz(a); }  // 0 for 0

// the `s` low bits of v, ones' complement for negative v (jchuff.c)
__device__ __forceinline__ uint32_t magnitude(int v, uint32_t s) { return (uint32_t)(v < 0 ? v - 1 : v) & ((1u << s) - 1u); }

// ---- jpeg_transform ------------------------------------------------------------------------------------------
// jfdctint.c jpeg_fdct_islow, one pass over 8 values `stride` apart (FINAL: the column pass)
template <bool FINAL>
__device__ __forceinline__ void fdct_pass(int *d, int stride) {
    constexpr int CB = 13, P1 = 2, SH = FINAL ? CB + P1 : CB - P1;
    const int t0 = d[0] + d[7 * stride], t7 = d[0] - d[7 * stride];
    const int t1 = d[stride] + d[6 * stride], t6 = d[stride] - d[6 * stride];
    const int t2 = d[2 * stride] + d[5 * stride], t5 = d[2 * stride] - d[5 * stride];
    const int t3 = d[3 * stride] + d[4 * stride], t4 = d[3 * stride] - d[4 * stride];
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    if (FINAL) {
        d[0] = (t10 + t11 + (1 << (P1 - 1))) >> P1;
        d[4 * stride] = (t10 - t11 + (1 << (P1 - 1))) >> P1;
    } else {
        d[0] = (t10 + t11) * (1 << P1);
        d[4 * stride] = (t10 - t11) * (1 << P1);
    }
    const int r = 1 << (SH - 1);
    int z1 = (t12 + t13) * 4433;
    d[2 * stride] = (z1 + t13 * 6270 + r) >> SH;
    d[6 * stride] = (z1 - t12 * 15137 + r) >> SH;
    z1 = t4 + t7;
    int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const int z5 = (z3 + z4) * 9633;
    z1 *= -7373, z2 *= -20995, z3 = z3 * -16069 + z5, z4 = z4 * -3196 + z5;
    d[7 * stride] = (t4 * 2446 + z1 + z3 + r) >> SH;
    d[5 * stride] = (t5 * 16819 + z2 + z4 + r) >> SH;
    d[3 * stride] = (t6 * 25172 + z2 + z3 + r) >> SH;
    d[stride] = (t7 * 12299 + z1 + z4 + r) >> SH;
}

// one 16-byte-or-narrower group of a lane's 8 pixels: RGBA words of columns x0 .. x0+7 of `row`, replicated past
// the last column
__device__ __forceinline__ void load_pixels(const uint8_t *row, uint32_t x0, uint32_t width, bool vec, uint32_t px[8]) {
    if (vec && x0 + 8u <= width) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(row + 4u * x0));
        const uint4 b = __ldg(reinterpret_cast<const uint4 *>(row + 4u * x0 + 16u));
        px[0] = a.x, px[1] = a.y, px[2] = a.z, px[3] = a.w, px[4] = b.x, px[5] = b.y, px[6] = b.z, px[7] = b.w;
    } else {
#pragma unroll
        for (uint32_t k = 0; k < 8; k++) {
            const uint8_t *p = row + 4u * min(x0 + k, width - 1u);
            px[k] = (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16;
        }
    }
}

// One warp per MCU, T_WARPS MCUs per CTA.
__global__ void __launch_bounds__(T_WARPS * 32) jpeg_transform(const uint8_t *__restrict__ rgba, size_t pitch,
                                                                uint32_t width, uint32_t height, bool vec,
                                                                const __grid_constant__ Tables tab, Scratch sc) {
    __shared__ int s_blk[T_WARPS][6][64];         // Y00 Y01 Y10 Y11 Cb Cr, natural order
    __shared__ uint8_t s_c[T_WARPS][2][16][16];   // full-resolution Cb, Cr
    __shared__ uint8_t s_size[2][256];            // AC code lengths
    __shared__ uint16_t s_div[2][64];
    for (uint32_t i = threadIdx.x; i < 512; i += blockDim.x) s_size[i >> 8][i & 255] = (uint8_t)(tab.ac[i >> 8][i & 255] >> 16);
    for (uint32_t i = threadIdx.x; i < 128; i += blockDim.x) s_div[i >> 6][i & 63] = tab.div[i >> 6][i & 63];
    __syncthreads();

    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t mcus = (width + 15u) / 16u, rows = (height + 15u) / 16u;
    const uint32_t mcu = blockIdx.x * T_WARPS + warp;
    if (mcu >= mcus * rows) return;
    const uint32_t mx = mcu % mcus, my = mcu / mcus;
    int(*blk)[64] = s_blk[warp];

    // pixels: lane = row r (0..15), half h; rows past the image repeat its last row
    {
        const uint32_t r = lane >> 1, c0 = (lane & 1u) * 8u;
        const uint8_t *row = rgba + (size_t)min(my * 16u + r, height - 1u) * pitch;
        uint32_t px[8];
        load_pixels(row, mx * 16u + c0, width, vec, px);
        int *yb = blk[(r >> 3) * 2u + (c0 >> 3)] + (r & 7u) * 8u;
#pragma unroll
        for (uint32_t k = 0; k < 8; k++) {  // jccolor.c rgb_ycc_convert
            const int R = px[k] & 255u, G = (px[k] >> 8) & 255u, B = (px[k] >> 16) & 255u;
            yb[k] = ((19595 * R + 38470 * G + 7471 * B + 32768) >> 16) - 128;
            s_c[warp][0][r][c0 + k] = (uint8_t)((-11059 * R - 21709 * G + 32768 * B + (128 << 16) + 32767) >> 16);
            s_c[warp][1][r][c0 + k] = (uint8_t)((32768 * R - 27439 * G - 5329 * B + (128 << 16) + 32767) >> 16);
        }
    }
    __syncwarp();
    // jcsample.c h2v2_downsample (bias 1, 2 alternating along the row); chroma rows past the image's (h + 1) / 2
    // repeat its last chroma row (jcprepct.c pads each component after downsampling)
    const uint32_t last_crow = (height + 1u) / 2u - 1u;
#pragma unroll
    for (uint32_t s = 0; s < 2; s++) {
        const uint32_t i = lane + 32u * s, oy = min(my * 8u + (i >> 3), last_crow) - my * 8u, ox = i & 7u;
#pragma unroll
        for (uint32_t c = 0; c < 2; c++) {
            const uint8_t *a = s_c[warp][c][2u * oy] + 2u * ox, *b = s_c[warp][c][2u * oy + 1u] + 2u * ox;
            blk[4 + c][i] = (int)((a[0] + a[1] + b[0] + b[1] + 1u + (ox & 1u)) >> 2) - 128;
        }
    }
    __syncwarp();
    // FDCT: 48 rows, then 48 columns
    for (uint32_t t = lane; t < 48u; t += 32u) fdct_pass<false>(blk[t >> 3] + (t & 7u) * 8u, 1);
    __syncwarp();
    for (uint32_t t = lane; t < 48u; t += 32u) fdct_pass<true>(blk[t >> 3] + (t & 7u), 8);
    __syncwarp();

    // quantise (round half away from zero by 8 * qtbl), lane holds zig-zag positions lane and lane + 32
    int q[6][2];
#pragma unroll
    for (uint32_t b = 0; b < 6; b++) {
#pragma unroll
        for (uint32_t s = 0; s < 2; s++) {
            const uint32_t nat = c_zigzag[lane + 32u * s];
            const int v = blk[b][nat], d = s_div[b >= 4][nat];
            const int m = ((v < 0 ? -v : v) + (d >> 1)) / d;
            q[b][s] = v < 0 ? -m : m;
        }
    }
    // jccoefct.c dummy blocks: a luma block past the image's last block column or row is AC zero with the DC of the
    // block before it in the MCU (for a bottom one, of Y01, itself a dummy copying Y00 when past the last column)
    const bool right = mx * 2u + 1u >= (width + 7u) / 8u, bottom = my * 2u + 1u >= (height + 7u) / 8u;
    if (right) {
        const int dc = __shfl_sync(FULL, q[0][0], 0);
        q[1][0] = lane == 0 ? dc : 0, q[1][1] = 0;
    }
    if (bottom) {
        const int dc = __shfl_sync(FULL, q[1][0], 0);
        q[2][0] = q[3][0] = lane == 0 ? dc : 0, q[2][1] = q[3][1] = 0;
    } else if (right) {
        const int dc = __shfl_sync(FULL, q[2][0], 0);
        q[3][0] = lane == 0 ? dc : 0, q[3][1] = 0;
    }

    // store, and each block's AC bits: a coefficient's run is the distance to the previous nonzero one (the DC
    // position counts as one), ZRL per 16 zeros, then its code and its bits; EOB unless position 63 is nonzero
    const size_t blk0 = (size_t)mcu * 6u;
#pragma unroll
    for (uint32_t b = 0; b < 6; b++) {
        int16_t *dst = sc.coef + (blk0 + b) * 64u;
        dst[lane] = (int16_t)q[b][0];
        dst[lane + 32u] = (int16_t)q[b][1];
        const uint32_t t = b >= 4;
        const unsigned long long m = (unsigned long long)__ballot_sync(FULL, q[b][0] != 0) |
                                     (unsigned long long)__ballot_sync(FULL, q[b][1] != 0) << 32 | 1ull;
        const uint32_t zrl = s_size[t][0xF0];
        uint32_t cost = 0;
#pragma unroll
        for (uint32_t s = 0; s < 2; s++) {
            const uint32_t z = lane + 32u * s;
            const int v = q[b][s];
            if (z >= 1u && v != 0) {
                const uint32_t prev = 63u - __clzll(m & ((1ull << z) - 1ull)), run = z - prev - 1u;
                const uint32_t n = nbits(v < 0 ? -v : v);
                cost += (run >> 4) * zrl + s_size[t][(run & 15u) << 4 | n] + n;
            }
        }
        if (lane == 0 && !(m >> 63)) cost += s_size[t][0];
#pragma unroll
        for (uint32_t d = 16; d; d >>= 1) cost += __shfl_xor_sync(FULL, cost, d);
        if (lane == 0) sc.acbits[blk0 + b] = cost;
    }
}

// ---- jpeg_encode_rows ----------------------------------------------------------------------------------------
// Exclusive scan of v over the CTA (blockDim.x = 32 * warps); *total gets the sum.  s_part holds 33 words.
__device__ __forceinline__ uint32_t block_scan(uint32_t v, uint32_t *s_part, uint32_t *total) {
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, warps = blockDim.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(FULL, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) s_part[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < warps ? s_part[lane] : 0u, wi = w;
#pragma unroll
        for (uint32_t d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(FULL, wi, d);
            if (lane >= d) wi += o;
        }
        if (lane < warps) s_part[lane] = wi - w;
        if (lane == 31) s_part[32] = wi;
    }
    __syncthreads();
    const uint32_t r = s_part[warp] + inc - v;
    *total = s_part[32];
    __syncthreads();  // s_part is reused
    return r;
}

// `n` (1..32) bits of `v` at bit `pos` of the MSB-first word stream
__device__ __forceinline__ void put_bits(uint32_t *stage, uint32_t pos, uint32_t v, uint32_t n) {
    const uint32_t w = pos >> 5, sh = pos & 31u;
    const unsigned long long x = (unsigned long long)v << (64u - sh - n);
    atomicOr(&stage[w], (uint32_t)(x >> 32));
    if (sh + n > 32u) atomicOr(&stage[w + 1], (uint32_t)x);
}

// The block before block i of a row in coding order with the same component, or -1 (the row's DC predictions
// start at 0): Y00 Y01 Y10 Y11 of an MCU follow each other, Cb and Cr follow the previous MCU's.
__device__ __forceinline__ int prev_same(uint32_t i) {
    const uint32_t b = i % 6u;
    if (b >= 1u && b <= 3u) return (int)i - 1;
    if (i < 6u) return -1;
    return b == 0 ? (int)i - 3 : (int)i - 6;
}

// One CTA per MCU row.
__global__ void __launch_bounds__(E_THREADS) jpeg_encode_rows(uint32_t width, const __grid_constant__ Tables tab,
                                                              Scratch sc) {
    __shared__ uint32_t s_dc[2][12], s_ac[2][256];
    __shared__ uint32_t s_part[33];
    for (uint32_t i = threadIdx.x; i < 512; i += blockDim.x) s_ac[i >> 8][i & 255] = tab.ac[i >> 8][i & 255];
    if (threadIdx.x < 24) s_dc[threadIdx.x / 12][threadIdx.x % 12] = tab.dc[threadIdx.x / 12][threadIdx.x % 12];
    __syncthreads();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t n = (width + 15u) / 16u * 6u;  // blocks in the row
    const size_t base = (size_t)blockIdx.x * n;
    const int16_t *coef = sc.coef + base * 64u;
    uint32_t *stage = sc.stage + (size_t)blockIdx.x * sc.slot_words;

    // each block's first bit: DC code and bits, plus its AC bits
    uint32_t bits = 0;
    for (uint32_t c = 0; c < n; c += blockDim.x) {
        const uint32_t i = c + threadIdx.x;
        uint32_t v = 0;
        if (i < n) {
            const int p = prev_same(i);
            const int diff = coef[(size_t)i * 64u] - (p < 0 ? 0 : coef[(size_t)p * 64u]);
            const uint32_t s = nbits(diff < 0 ? -diff : diff);
            v = (s_dc[i % 6u >= 4u][s] >> 16) + s + sc.acbits[base + i];
        }
        uint32_t total;
        const uint32_t off = bits + block_scan(v, s_part, &total);
        if (i < n) sc.boff[base + i] = off;
        bits += total;
    }
    // the segment's words start at zero, its padding is 1-bits
    const uint32_t pad = (8u - (bits & 7u)) & 7u, words = (bits + pad + 31u) / 32u;
    for (uint32_t w = threadIdx.x; w < words; w += blockDim.x) stage[w] = 0;
    __syncthreads();
    if (threadIdx.x == 0 && pad) atomicOr(&stage[bits >> 5], ((1u << pad) - 1u) << (32u - (bits & 31u) - pad));

    // one warp per block: lane holds zig-zag positions lane and lane + 32; each coefficient's codes (ZRLs, then
    // the run/size code and the bits) are placed by a warp scan of their lengths
    for (uint32_t i = warp; i < n; i += blockDim.x >> 5) {
        const uint32_t t = i % 6u >= 4u;
        const int16_t *cb = coef + (size_t)i * 64u;
        const int v0 = cb[lane], v1 = cb[lane + 32u];
        const unsigned long long m = (unsigned long long)__ballot_sync(FULL, v0 != 0) |
                                     (unsigned long long)__ballot_sync(FULL, v1 != 0) << 32 | 1ull;
        const uint32_t zrl = s_ac[t][0xF0], zrl_n = zrl >> 16;
        uint32_t code[2], len[2], nz[2], cost[2];
#pragma unroll
        for (uint32_t s = 0; s < 2; s++) {
            const uint32_t z = lane + 32u * s;
            const int v = s ? v1 : v0;
            code[s] = len[s] = nz[s] = 0;
            if (z == 0) {
                const int p = prev_same(i);
                const int diff = v - (p < 0 ? 0 : coef[(size_t)p * 64u]);
                const uint32_t sz = nbits(diff < 0 ? -diff : diff), h = s_dc[t][sz];
                code[s] = (h & 0xffffu) << sz | magnitude(diff, sz), len[s] = (h >> 16) + sz;
            } else if (v != 0) {
                const uint32_t prev = 63u - __clzll(m & ((1ull << z) - 1ull)), run = z - prev - 1u;
                const uint32_t sz = nbits(v < 0 ? -v : v), h = s_ac[t][(run & 15u) << 4 | sz];
                nz[s] = run >> 4;
                code[s] = (h & 0xffffu) << sz | magnitude(v, sz), len[s] = (h >> 16) + sz;
            }
            cost[s] = nz[s] * zrl_n + len[s];
        }
        uint32_t inc0 = cost[0], inc1 = cost[1];
#pragma unroll
        for (uint32_t d = 1; d < 32; d <<= 1) {
            const uint32_t o0 = __shfl_up_sync(FULL, inc0, d), o1 = __shfl_up_sync(FULL, inc1, d);
            if (lane >= d) inc0 += o0, inc1 += o1;
        }
        const uint32_t t0 = __shfl_sync(FULL, inc0, 31), t1 = __shfl_sync(FULL, inc1, 31);
        const uint32_t start = sc.boff[base + i];
        uint32_t pos[2] = {start + inc0 - cost[0], start + t0 + inc1 - cost[1]};
#pragma unroll
        for (uint32_t s = 0; s < 2; s++) {
            for (uint32_t k = 0; k < nz[s]; k++) put_bits(stage, pos[s] + k * zrl_n, zrl & 0xffffu, zrl_n);
            if (len[s]) put_bits(stage, pos[s] + nz[s] * zrl_n, code[s], len[s]);
        }
        if (lane == 0 && !(m >> 63)) put_bits(stage, start + t0 + t1, s_ac[t][0] & 0xffffu, s_ac[t][0] >> 16);
    }
    __syncthreads();

    // the segment's bytes and its 0xFF bytes
    const uint32_t bytes = (bits + pad) / 8u;
    uint32_t ff = 0;
    for (uint32_t w = threadIdx.x; w < words; w += blockDim.x) {
        const uint32_t x = stage[w];
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) ff += (4u * w + k < bytes && ((x >> (24u - 8u * k)) & 255u) == 255u);
    }
    uint32_t total;
    block_scan(ff, s_part, &total);
    if (threadIdx.x == 0) sc.rows[blockIdx.x] = make_uint2(bytes, total);
}

// ---- jpeg_assemble -------------------------------------------------------------------------------------------
// One CTA per MCU row.
__global__ void __launch_bounds__(A_THREADS) jpeg_assemble(uint32_t height, const __grid_constant__ Header hdr,
                                                           Scratch sc, uint8_t *__restrict__ out,
                                                           unsigned long long *len_word) {
    __shared__ unsigned long long s_red[A_THREADS / 32];
    __shared__ uint32_t s_part[33];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t row = blockIdx.x, rows = (height + 15u) / 16u;
    // this row's place: the header, then every earlier row's stuffed bytes and RST marker
    unsigned long long acc = 0;
    for (uint32_t j = threadIdx.x; j < row; j += blockDim.x) acc += sc.rows[j].x + sc.rows[j].y + 2u;
    for (uint32_t d = 16; d; d >>= 1) acc += __shfl_xor_sync(FULL, acc, d);
    if (lane == 0) s_red[warp] = acc;
    __syncthreads();
    unsigned long long off = HEADER_BYTES;
    for (uint32_t w = 0; w < A_THREADS / 32; w++) off += s_red[w];

    if (row == 0)
        for (uint32_t k = threadIdx.x; k < HEADER_BYTES; k += blockDim.x) out[k] = hdr.b[k];
    // the segment, a 0x00 after every 0xFF: a thread per word, placed by a scan of the words' 0xFF counts
    const uint2 seg = sc.rows[row];
    const uint32_t *stage = sc.stage + (size_t)row * sc.slot_words, words = (seg.x + 3u) / 4u;
    uint8_t *dst = out + off;
    uint32_t carry = 0;
    for (uint32_t c = 0; c < words; c += blockDim.x) {
        const uint32_t w = c + threadIdx.x;
        const uint32_t x = w < words ? stage[w] : 0u, nb = w < words ? min(4u, seg.x - 4u * w) : 0u;
        uint32_t ff = 0;
        for (uint32_t k = 0; k < nb; k++) ff += ((x >> (24u - 8u * k)) & 255u) == 255u;
        uint32_t total;
        uint32_t p = 4u * w + carry + block_scan(ff, s_part, &total);
        for (uint32_t k = 0; k < nb; k++) {
            const uint8_t byte = (uint8_t)(x >> (24u - 8u * k));
            dst[p++] = byte;
            if (byte == 0xFF) dst[p++] = 0;
        }
        carry += total;
    }
    if (threadIdx.x == 0) {
        uint8_t *end = dst + seg.x + seg.y;
        end[0] = 0xFF;
        if (row + 1u < rows) {
            end[1] = (uint8_t)(0xD0u + (row & 7u));
        } else {
            end[1] = 0xD9;
            *len_word = off + seg.x + seg.y + 2u;
        }
    }
}

Scratch scratch_at(const Layout &l, void *scratch) {
    uint8_t *p = static_cast<uint8_t *>(scratch);
    Scratch sc;
    sc.coef = reinterpret_cast<int16_t *>(p);
    p += l.coef_bytes;
    sc.acbits = reinterpret_cast<uint32_t *>(p);
    p += l.acbits_bytes;
    sc.boff = reinterpret_cast<uint32_t *>(p);
    p += l.boff_bytes;
    sc.stage = reinterpret_cast<uint32_t *>(p);
    p += l.stage_bytes;
    sc.rows = reinterpret_cast<uint2 *>(p);
    sc.slot_words = l.slot_words;
    return sc;
}

// jcparam.c jpeg_set_quality(quality, force_baseline = TRUE), jchuff.c jpeg_make_c_derived_tbl
void tables_of(int quality, Tables *t, uint8_t qtbl[2][64]) {
    memset(t, 0, sizeof(*t));
    const int scale = quality < 50 ? 5000 / quality : 200 - 2 * quality;
    for (int c = 0; c < 2; c++)
        for (int k = 0; k < 64; k++) {
            long v = ((long)k_base_quant[c][k] * scale + 50) / 100;
            v = v < 1 ? 1 : v > 255 ? 255 : v;
            qtbl[c][k] = (uint8_t)v;
            t->div[c][k] = (uint16_t)(8 * v);
        }
    for (int h = 0; h < 4; h++) {
        const uint8_t *vals = h & 1 ? k_ac_vals[h >> 1] : k_dc_vals;
        uint32_t *dst = h & 1 ? t->ac[h >> 1] : t->dc[h >> 1];
        uint32_t code = 0, k = 0;
        for (uint32_t len = 1; len <= 16; len++, code <<= 1)
            for (uint32_t i = 0; i < k_bits[h][len - 1]; i++, k++, code++) dst[vals[k]] = len << 16 | code;
    }
}

void header_of(uint32_t width, uint32_t height, const uint8_t qtbl[2][64], Header *hdr) {
    uint8_t *p = hdr->b;
    auto marker = [&](uint8_t m, uint32_t len) { *p++ = 0xFF, *p++ = m, *p++ = (uint8_t)(len >> 8), *p++ = (uint8_t)len; };
    *p++ = 0xFF, *p++ = 0xD8;
    marker(0xE0, 16);  // JFIF 1.01, no units, density 1:1, no thumbnail
    const uint8_t jfif[14] = {'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0};
    memcpy(p, jfif, 14), p += 14;
    for (int c = 0; c < 2; c++) {
        marker(0xDB, 67);
        *p++ = (uint8_t)c;
        for (int z = 0; z < 64; z++) *p++ = qtbl[c][k_zigzag[z]];
    }
    marker(0xC0, 17);
    const uint8_t sof[15] = {8, (uint8_t)(height >> 8), (uint8_t)height, (uint8_t)(width >> 8), (uint8_t)width, 3,
                             1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1};
    memcpy(p, sof, 15), p += 15;
    const uint8_t classes[4] = {0x00, 0x10, 0x01, 0x11};
    for (int h = 0; h < 4; h++) {
        const uint32_t n = h & 1 ? 162u : 12u;
        marker(0xC4, 2 + 1 + 16 + n);
        *p++ = classes[h];
        memcpy(p, k_bits[h], 16), p += 16;
        memcpy(p, h & 1 ? k_ac_vals[h >> 1] : k_dc_vals, n), p += n;
    }
    const uint32_t interval = (width + 15) / 16;  // one MCU row
    marker(0xDD, 4);
    *p++ = (uint8_t)(interval >> 8), *p++ = (uint8_t)interval;
    marker(0xDA, 12);
    const uint8_t sos[10] = {3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0};
    memcpy(p, sos, 10), p += 10;
}

}  // namespace

size_t rt_jpeg_bound_bytes(uint32_t width, uint32_t height) {
    const Layout l = layout_of(width, height);
    return HEADER_BYTES + (size_t)l.rows * (2 * ((size_t)l.mcus * 6 * BLOCK_BITS / 8 + 1) + 2) + 2;
}

size_t rt_jpeg_scratch_bytes(uint32_t width, uint32_t height) {
    const Layout l = layout_of(width, height);
    return l.coef_bytes + l.acbits_bytes + l.boff_bytes + l.stage_bytes + l.rows_bytes;
}

cudaError_t rt_launch_jpeg_encode(const uint8_t *rgba, size_t pitch, uint32_t width, uint32_t height, int quality,
                                  void *scratch, uint8_t *out, unsigned long long *len_word, cudaStream_t stream) {
    if (width == 0 || height == 0 || quality < 1 || quality > 100) return cudaErrorInvalidValue;
    const Layout l = layout_of(width, height);
    const Scratch sc = scratch_at(l, scratch);
    Tables tab;
    uint8_t qtbl[2][64];
    tables_of(quality, &tab, qtbl);
    Header hdr;
    header_of(width, height, qtbl, &hdr);
    const bool vec = ((uintptr_t)rgba & 15u) == 0 && (pitch & 15u) == 0;
    const uint32_t mcus = l.mcus * l.rows;
    jpeg_transform<<<(mcus + T_WARPS - 1) / T_WARPS, T_WARPS * 32, 0, stream>>>(rgba, pitch, width, height, vec, tab, sc);
    jpeg_encode_rows<<<l.rows, E_THREADS, 0, stream>>>(width, tab, sc);
    jpeg_assemble<<<l.rows, A_THREADS, 0, stream>>>(height, hdr, sc, out, len_word);
    return cudaGetLastError();
}
