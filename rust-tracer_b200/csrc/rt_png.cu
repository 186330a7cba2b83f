// rt_png.cu -- PNG files encoded on the device (rt_encode_png, rt_render_sweep_png).
//
// The layout is fixed so that there is exactly one byte string per image (tests/_png_ref.py is the reference
// encoder; DESIGN.md "PNG output" explains the choices):
//   signature, IHDR (8-bit RGB, colour type 2, no interlace), IDAT "78 01" (zlib header),
//   one IDAT per band of 16 rows, a band being its rows' pieces back to back, each piece a non-final
//   fixed-Huffman block of the raw row (filter byte 0 + RGB) ended by end-of-block and an empty non-final stored
//   block (so every piece is byte-aligned and independent of its neighbours),
//   IDAT "03 00" (final empty fixed block) + Adler-32, IEND.
// Parse rule of a row: raw byte i is "repeated" when i >= 4 and row[i] == row[i-3]; a maximal run of R repeated
// bytes is floor(R/258) matches of 258, then one match of R mod 258 if that is >= 3, else R mod 258 literals; every
// match has distance 3; every other byte is a literal.  Token lengths are therefore known in closed form per run.
//
// Two launches: png_encode_rows (one CTA per band, one warp per row: run masks, token bit offsets by warp scans,
// bits packed in shared memory and flushed to a global staging slot per row, the piece's CRC-32 and Adler-32
// partials), then the assemble kernel (one CTA per band: the chunk's place from a scan of the band sizes, the copy of
// its pieces into the file; CTA 0 writes the header, one more CTA the last zlib chunk, IEND and the length).  Its one
// body, assemble<ANIMATED>, is png_assemble for a PNG file and apng_assemble for one frame of an animated PNG
// (rt_encode_apng_frame, rt_render_sweep_apng): the same zlib stream, framed as that frame's piece of the animation
// (DESIGN.md "Animated PNG").
#include "rt_png.h"

namespace {

constexpr uint32_t BAND = 16;          // rows per IDAT chunk (the multi-GPU row-block unit)
constexpr uint32_t WARPS = BAND;       // one warp per row of the band
constexpr uint32_t ADLER_MOD = 65521u;
constexpr uint32_t FULL = 0xffffffffu;
constexpr uint32_t HEADER_BYTES = 8 + 25 + 14;  // signature, IHDR, IDAT(78 01)
constexpr uint32_t TRAILER_BYTES = 18 + 12;     // IDAT(03 00 + Adler-32), IEND
constexpr uint32_t ACTL_BYTES = 12 + 8, FCTL_BYTES = 12 + 26;

__constant__ uint16_t c_len_base[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23, 27,
                                        31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};

struct Scratch {
    uint32_t *stage;  // per row: slot_words words of token bits (LSB-first)
    uint32_t *masks;  // per row: mask_stride words, bit p = raw byte p is repeated
    uint4 *rows;      // per row: {bits, crc32 of the piece, sum of bytes mod 65521, weighted sum mod 65521}
    uint2 *bands;     // per band: {data bytes, crc32 of "IDAT" + data}
    uint32_t slot_words, mask_stride;
};

struct Layout {
    uint32_t n, bands, slot_words, mask_stride;
    size_t stage_bytes, mask_bytes, rows_bytes, bands_bytes;
};

size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

Layout layout_of(uint32_t width, uint32_t height) {
    Layout l;
    l.n = 1 + 3 * width;
    l.bands = (height + BAND - 1) / BAND;
    l.slot_words = (uint32_t)round_up((3 + 9ull * l.n + 31) / 32, 32);  // 9 bits per byte at most, 128-byte slots
    l.mask_stride = (uint32_t)round_up((l.n + 31) / 32, 32);
    l.stage_bytes = (size_t)height * l.slot_words * 4;
    l.mask_bytes = (size_t)height * l.mask_stride * 4;
    l.rows_bytes = round_up((size_t)height * sizeof(uint4), 128);
    l.bands_bytes = round_up((size_t)l.bands * sizeof(uint2), 128);
    return l;
}

// ---- CRC-32 (zlib's polynomial, reflected) -----------------------------------------------------------------
__device__ __forceinline__ uint32_t crc_table_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = (c & 1u) ? 0xedb88320u ^ (c >> 1) : c >> 1;
    return c;
}

// a * b mod P in zlib's reflected representation (crc32_combine's multmodp)
__device__ uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (uint32_t m = 1u << 31; m; m >>= 1) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1u)) == 0) break;
        }
        b = (b & 1u) ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}

// crc32(A || B) from crc32(A), crc32(B) and |B| (zlib's crc32_combine); x2n[k] = x^(2^k) mod P
__device__ uint32_t crc_combine(uint32_t crc_a, uint32_t crc_b, uint32_t len_b, const uint32_t *x2n) {
    uint32_t p = 1u << 31, k = 3;  // x^0; bytes -> bits is 2^3
    for (uint32_t n = len_b; n; n >>= 1, k++)
        if (n & 1u) p = multmodp(x2n[k & 31], p);
    return multmodp(p, crc_a) ^ crc_b;
}

__device__ uint32_t crc_bytes(uint32_t c, const uint8_t *p, uint32_t n, const uint32_t *table) {
    for (uint32_t i = 0; i < n; i++) c = table[(c ^ p[i]) & 255u] ^ (c >> 8);
    return c;
}

// Both kernels: the byte table and the x^(2^k) table in shared memory.
__device__ void init_crc_tables(uint32_t *table, uint32_t *x2n) {
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) table[i] = crc_table_entry(i);
    if (threadIdx.x < 32) {
        uint32_t p = 1u << 30;  // x^1
        for (uint32_t k = 0; k < threadIdx.x; k++) p = multmodp(p, p);
        x2n[threadIdx.x] = p;
    }
}

__device__ __forceinline__ void put_be32(uint8_t *p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24), p[1] = (uint8_t)(v >> 16), p[2] = (uint8_t)(v >> 8), p[3] = (uint8_t)v;
}

// A chunk of `n` data bytes already at p + 8: length, type and CRC around them.
__device__ void write_chunk(uint8_t *p, const char *type, uint32_t n, const uint32_t *table) {
    put_be32(p, n);
    for (int k = 0; k < 4; k++) p[4 + k] = (uint8_t)type[k];
    put_be32(p + 8 + n, ~crc_bytes(0xffffffffu, p + 4, 4 + n, table));
}

// ---- fixed Huffman codes (RFC 1951 3.2.6), bit-reversed for the LSB-first stream --------------------------------
__device__ __forceinline__ uint32_t lit_bits(uint32_t v) { return v < 144u ? 8u : 9u; }

__device__ __forceinline__ uint32_t lit_code(uint32_t v) {
    return v < 144u ? __brev(0x30u + v) >> 24 : __brev(0x190u + v - 144u) >> 23;
}

// length L (3..258) + distance 3 (code 2, 5 bits): one token of at most 8 + 5 + 5 = 18 bits
__device__ uint32_t match_code(uint32_t L, uint32_t *bits) {
    int k = 28;
    while (c_len_base[k] > L) k--;
    const uint32_t sym = 257u + (uint32_t)k;
    uint32_t c, n;
    if (sym < 280u) c = __brev(sym - 256u) >> 25, n = 7;
    else c = __brev(0xC0u + sym - 280u) >> 24, n = 8;
    c |= (L - c_len_base[k]) << n;
    n += c_len_extra[k];
    c |= (__brev(2u) >> 27) << n;
    *bits = n + 5;
    return c;
}

__device__ __forceinline__ uint32_t raw_byte(const uint8_t *row, uint32_t p) {  // raw-row byte p >= 1
    const uint32_t q = p - 1u, x = q / 3u;
    return row[4u * x + (q - 3u * x)];
}

// Bytes of a row's piece: the staged token bits, zeros (end-of-block, the stored block's header, padding), then
// the stored block's LEN / NLEN 00 00 FF FF.
__device__ __forceinline__ uint32_t piece_bytes(uint32_t bits) { return (bits + 10u + 7u) / 8u + 4u; }

__device__ __forceinline__ uint32_t piece_byte(const uint8_t *staged, uint32_t bits, uint32_t len, uint32_t q) {
    return q < (bits + 7u) / 8u ? staged[q] : (q + 2u >= len ? 0xffu : 0u);
}

// One CTA per band of 16 rows, one warp per row.
__global__ void __launch_bounds__(WARPS * 32) png_encode_rows(const uint8_t *__restrict__ rgba, size_t pitch,
                                                                uint32_t width, uint32_t height, Scratch sc) {
    __shared__ uint32_t s_table[256], s_x2n[32];
    __shared__ uint32_t s_buf[WARPS][64];  // a warp's pending output words
    __shared__ uint32_t s_len[WARPS], s_crc[WARPS];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    init_crc_tables(s_table, s_x2n);
    uint32_t *buf = s_buf[warp];
    buf[lane] = lane == 0 ? 2u : 0u;  // the row's block header: BFINAL 0, BTYPE 01 is bit value 2
    buf[lane + 32] = 0;
    __syncthreads();

    const uint32_t r = blockIdx.x * BAND + warp;
    if (r < height) {
        const uint8_t *row = rgba + (size_t)r * pitch;
        const uint32_t n = 1u + 3u * width, nw = (n + 31u) / 32u;
        uint32_t *mask = sc.masks + (size_t)r * sc.mask_stride;
        uint32_t *stage = sc.stage + (size_t)r * sc.slot_words;

        // pass 1: which raw bytes repeat the same channel of the previous pixel
#pragma unroll 4
        for (uint32_t k = 0; k < nw; k++) {
            const uint32_t p = k * 32u + lane;
            bool e = false;
            if (p >= 4u && p < n) {
                const uint32_t q = p - 1u, x = q / 3u, o = 4u * x + (q - 3u * x);
                e = row[o] == row[o - 4u];
            }
            const uint32_t m = __ballot_sync(FULL, e);
            if (lane == 0) mask[k] = m;
        }
        __syncwarp();

        // pass 2: token bit offsets (a run's whole length is charged to its first byte, so an exclusive scan gives
        // every literal's and every run's offset), the tokens, the Adler-32 partials
        const uint32_t code258 = (__brev(0xC5u) >> 24) | ((__brev(2u) >> 27) << 8);  // symbol 285 + distance 3
        uint32_t bits = 3;  // after the block header
        uint32_t base_word = 0;                        // stream word held in buf[0]
        uint32_t run_s = 0, run_len = 0, run_off = 0;  // the run reaching into this step from earlier ones
        uint32_t prev_eq = 0, prev_v = 0;
        unsigned long long sum = 0, wsum = 0;
        for (uint32_t k = 0; k < nw; k++) {
            const uint32_t p = k * 32u + lane;
            const bool valid = p < n;
            const uint32_t v = (valid && p) ? raw_byte(row, p) : 0u;
            const uint32_t m = mask[k];
            const bool eq = (m >> lane) & 1u;
            const bool start = eq && !(lane ? (m >> (lane - 1u)) & 1u : prev_eq);
            uint32_t R = 0, cost = 0;
            if (start) {  // the run ends at the first clear bit at or after p (bits past the row are clear)
                uint32_t wk = k, z = ~m & (FULL << lane);
                while (z == 0 && ++wk < nw) z = ~mask[wk];
                const uint32_t t = z ? min(wk * 32u + __ffs(z) - 1u, n) : n;
                R = t - p;
                const uint32_t q = R / 258u, rr = R - 258u * q;
                cost = 13u * q;
                if (rr >= 3u) {
                    uint32_t nb;
                    match_code(rr, &nb);
                    cost += nb;
                } else {
                    for (uint32_t i = t - rr; i < t; i++) cost += lit_bits(raw_byte(row, i));
                }
            } else if (valid && !eq) {
                cost = lit_bits(v);
            }
            uint32_t inc = cost;
#pragma unroll
            for (uint32_t d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_up_sync(FULL, inc, d);
                if (lane >= d) inc += o;
            }
            const uint32_t off = bits + inc - cost;
            // the run this byte belongs to: the highest run start at or below this lane, else the carried one
            const uint32_t starts = __ballot_sync(FULL, start);
            const uint32_t le = starts & (FULL >> (31u - lane));
            const int src = le ? 31 - __clz(le) : (int)lane;
            const uint32_t ss = __shfl_sync(FULL, p, src), sR = __shfl_sync(FULL, R, src), so = __shfl_sync(FULL, off, src);
            const uint32_t up_v = __shfl_up_sync(FULL, v, 1);
            const uint32_t vprev = lane ? up_v : prev_v;
            uint32_t code = 0, nb = 0, o = 0;
            if (valid && !eq) {
                code = lit_code(v), nb = lit_bits(v), o = off;
            } else if (eq) {
                const uint32_t rs = le ? ss : run_s, rl = le ? sR : run_len, ro = le ? so : run_off;
                const uint32_t j = p - rs, q = rl / 258u, tail = 258u * q, rr = rl - tail;
                if (j < tail) {
                    if (j % 258u == 0) code = code258, nb = 13, o = ro + 13u * (j / 258u);
                } else if (rr >= 3u) {
                    if (j == tail) code = match_code(rr, &nb), o = ro + 13u * q;
                } else {
                    code = lit_code(v), nb = lit_bits(v), o = ro + 13u * q + (j > tail ? lit_bits(vprev) : 0u);
                }
            }
            if (nb) {
                const uint32_t w = (o >> 5) - base_word, sh = o & 31u;
                atomicOr(&buf[w], code << sh);
                if (sh + nb > 32u) atomicOr(&buf[w + 1], code >> (32u - sh));
            }
            if (valid) sum += v, wsum += (unsigned long long)(n - p) * v;
            bits += __shfl_sync(FULL, inc, 31);
            if (starts) {
                const int hi = 31 - __clz(starts);
                run_s = __shfl_sync(FULL, p, hi), run_len = __shfl_sync(FULL, R, hi), run_off = __shfl_sync(FULL, off, hi);
            }
            prev_eq = m >> 31;
            prev_v = __shfl_sync(FULL, v, 31);
            // bits below `frontier` are final: everything, unless a run continues into the next step -- then up to
            // the token covering this step's last byte
            const uint32_t last = k * 32u + 31u;
            const uint32_t frontier = (prev_eq && run_s + run_len > last + 1u) ? run_off + 13u * ((last - run_s) / 258u) : bits;
            __syncwarp();
            if ((frontier >> 5) - base_word >= 32u) {
                stage[base_word + lane] = buf[lane];
                buf[lane] = buf[lane + 32];
                buf[lane + 32] = 0;
                base_word += 32u;
                __syncwarp();
            }
        }
        const uint32_t words = (bits + 31u) >> 5;
        for (uint32_t i = lane; base_word + i < words; i += 32u) stage[base_word + i] = buf[i];
        __syncwarp();

        // the piece's CRC-32: a slice per lane, combined across the warp
        const uint32_t len = piece_bytes(bits), slice = (len + 31u) / 32u;
        const uint32_t b0 = min(len, lane * slice), b1 = min(len, b0 + slice);
        const uint8_t *staged = reinterpret_cast<const uint8_t *>(stage);
        uint32_t c = 0xffffffffu;
        for (uint32_t q = b0; q < b1; q++) c = s_table[(c ^ piece_byte(staged, bits, len, q)) & 255u] ^ (c >> 8);
        c = ~c;
        uint32_t clen = b1 - b0;
        for (uint32_t d = 1; d < 32; d <<= 1) {
            const uint32_t oc = __shfl_down_sync(FULL, c, d), ol = __shfl_down_sync(FULL, clen, d);
            if ((lane & (2u * d - 1u)) == 0) c = crc_combine(c, oc, ol, s_x2n), clen += ol;
        }
        for (uint32_t d = 16; d; d >>= 1) {
            sum += __shfl_xor_sync(FULL, sum, d);
            wsum += __shfl_xor_sync(FULL, wsum, d);
        }
        if (lane == 0) {
            sc.rows[r] = make_uint4(bits, c, (uint32_t)(sum % ADLER_MOD), (uint32_t)(wsum % ADLER_MOD));
            s_len[warp] = len;
            s_crc[warp] = c;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // the band's chunk: data size and CRC-32 over "IDAT" + data
        const uint32_t rows = min(BAND, height - blockIdx.x * BAND);
        const uint8_t idat[4] = {'I', 'D', 'A', 'T'};
        uint32_t c = ~crc_bytes(0xffffffffu, idat, 4, s_table), d = 0;
        for (uint32_t w = 0; w < rows; w++) c = crc_combine(c, s_crc[w], s_len[w], s_x2n), d += s_len[w];
        sc.bands[blockIdx.x] = make_uint2(d, c);
    }
}

// ---- the assemble kernels' steps ------------------------------------------------------------------------------
// The offset of CTA b's chunk (`head` bytes, then every earlier band's chunk of `framing` +
// data bytes), and in s_rowoff the offsets of its rows' pieces within the chunk's data.
__device__ __forceinline__ unsigned long long chunk_offset(const Scratch &sc, uint32_t height, uint32_t b,
                                                           uint32_t framing, uint32_t head, unsigned long long *s_red,
                                                           uint32_t *s_rowoff) {
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t bands = (height + BAND - 1) / BAND;
    unsigned long long acc = 0;
    for (uint32_t i = threadIdx.x; i < b; i += blockDim.x) acc += framing + sc.bands[i].x;
    for (uint32_t d = 16; d; d >>= 1) acc += __shfl_xor_sync(FULL, acc, d);
    if (lane == 0) s_red[warp] = acc;
    if (threadIdx.x == 0) {
        const uint32_t rows = b < bands ? min(BAND, height - b * BAND) : 0u;
        s_rowoff[0] = 0;
        for (uint32_t w = 0; w < rows; w++) s_rowoff[w + 1] = s_rowoff[w] + piece_bytes(sc.rows[b * BAND + w].x);
    }
    __syncthreads();
    unsigned long long off = head;
    for (uint32_t w = 0; w < WARPS; w++) off += s_red[w];
    return off;
}

// Band b's pieces, one row per warp, to `dst` (the chunk's data).
__device__ __forceinline__ void copy_pieces(const Scratch &sc, uint32_t height, uint32_t b, uint8_t *dst,
                                            const uint32_t *s_rowoff) {
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t r = b * BAND + warp;
    if (r < height) {
        const uint32_t bits = sc.rows[r].x, len = piece_bytes(bits);
        const uint8_t *staged = reinterpret_cast<const uint8_t *>(sc.stage + (size_t)r * sc.slot_words);
        uint8_t *d = dst + s_rowoff[warp];
        for (uint32_t q = lane; q < len; q += 32u) d[q] = (uint8_t)piece_byte(staged, bits, len, q);
    }
}

// The PNG signature and IHDR at `out` (33 bytes).
__device__ __forceinline__ void write_signature_ihdr(uint8_t *out, uint32_t width, uint32_t height, const uint32_t *table) {
    const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
    for (int k = 0; k < 8; k++) out[k] = sig[k];
    uint8_t *ihdr = out + 8;
    put_be32(ihdr + 8, width);
    put_be32(ihdr + 12, height);
    ihdr[16] = 8, ihdr[17] = 2, ihdr[18] = 0, ihdr[19] = 0, ihdr[20] = 0;
    write_chunk(ihdr, "IHDR", 13, table);
}

// The zlib stream's Adler-32 (returned to thread 0) from the per-row partials.  Row r of n
// bytes starts at byte r*n of N = n*h, so b gains W_r + n*(h-1-r)*S_r, where S_r = sum of its bytes and
// W_r = sum of (n - k) * byte k.
__device__ __forceinline__ uint32_t adler_of_rows(const Scratch &sc, uint32_t width, uint32_t height,
                                                  unsigned long long *s_red, unsigned long long *s_red2) {
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t n = 1u + 3u * width, nm = n % ADLER_MOD;
    unsigned long long sa = 0, sb = 0;
    for (uint32_t r = threadIdx.x; r < height; r += blockDim.x) {
        const uint4 ri = sc.rows[r];
        const unsigned long long wgt = (unsigned long long)nm * ((height - 1u - r) % ADLER_MOD) % ADLER_MOD;
        sa += ri.z;
        sb += (ri.w + wgt * ri.z) % ADLER_MOD;
    }
    for (uint32_t d = 16; d; d >>= 1) sa += __shfl_xor_sync(FULL, sa, d), sb += __shfl_xor_sync(FULL, sb, d);
    __syncthreads();  // s_red is reused
    if (lane == 0) s_red[warp] = sa, s_red2[warp] = sb;
    __syncthreads();
    if (threadIdx.x != 0) return 0;
    unsigned long long a = 1, bb = (unsigned long long)n * height % ADLER_MOD;
    for (uint32_t w = 0; w < WARPS; w++) a += s_red[w], bb += s_red2[w];
    a %= ADLER_MOD, bb %= ADLER_MOD;
    return (uint32_t)((bb << 16) | a);
}

// The file (ANIMATED = false) or frame `frame`'s payload of an n_frames animated PNG (ANIMATED, delay = delay_num << 16
// | delay_den).  CTA b < bands: band b's chunk, CTA 0 also the header; CTA `bands`: the last zlib chunk, IEND and the
// length.  A file is signature, IHDR, the IDAT chunks, IEND.  A payload is frame 0: signature, IHDR, acTL, fcTL 0, then
// the frame's IDAT chunks exactly as its file has them; frame f >= 1: fcTL s_f, then the same C = bands + 2 chunks as
// fdAT, chunk k carrying sequence number s_f + 1 + k before its data, where s_f = 1 + (f - 1)(C + 1).  The last frame
// also ends with IEND.  The animation is the payloads in frame order, so no frame depends on another.
template <bool ANIMATED>
__device__ __forceinline__ void assemble(uint32_t width, uint32_t height, const Scratch &sc, uint32_t frame,
                                         uint32_t n_frames, uint32_t delay, uint8_t *__restrict__ out,
                                         unsigned long long *len_word) {
    __shared__ uint32_t s_table[256], s_x2n[32];
    __shared__ unsigned long long s_red[WARPS], s_red2[WARPS];
    __shared__ uint32_t s_rowoff[BAND + 1];
    const uint32_t b = blockIdx.x;
    const uint32_t bands = (height + BAND - 1) / BAND;
    const bool first = !ANIMATED || frame == 0;  // the payload starts the file
    const uint32_t seq_bytes = first ? 0u : 4u;  // an fdAT's sequence number, before the data
    const uint32_t fctl_seq = first ? 0u : 1u + (frame - 1u) * (bands + 3u);
    init_crc_tables(s_table, s_x2n);
    const uint32_t head = (first ? 8u + 25u : 0u) + (ANIMATED ? (first ? ACTL_BYTES : 0u) + FCTL_BYTES : 0u) + 14u + seq_bytes;
    const unsigned long long off = chunk_offset(sc, height, b, 12u + seq_bytes, head, s_red, s_rowoff);

    if (b < bands) {
        copy_pieces(sc, height, b, out + off + 8 + seq_bytes, s_rowoff);
        if (threadIdx.x == 0) {
            const uint2 band = sc.bands[b];
            uint8_t *c = out + off;
            put_be32(c, band.x + seq_bytes);
            if (first) {
                c[4] = 'I', c[5] = 'D', c[6] = 'A', c[7] = 'T';
                put_be32(c + 8 + band.x, band.y);
            } else {
                // crc("fdAT" seq data) = crc("IDAT" data) ^ x^(8 |data|) (crc("IDAT") ^ crc("fdAT" seq)): the band's
                // CRC is reused instead of reading the data again
                c[4] = 'f', c[5] = 'd', c[6] = 'A', c[7] = 'T';
                put_be32(c + 8, fctl_seq + 2u + b);
                const uint8_t idat[4] = {'I', 'D', 'A', 'T'};
                const uint32_t diff = ~crc_bytes(0xffffffffu, idat, 4, s_table) ^ ~crc_bytes(0xffffffffu, c + 4, 8, s_table);
                put_be32(c + 12 + band.x, band.y ^ crc_combine(diff, 0u, band.x, s_x2n));
            }
        }
        if (b == 0 && threadIdx.x == 0) {
            uint8_t *p = out;
            if (first) {
                write_signature_ihdr(p, width, height, s_table);
                p += 33;
                if constexpr (ANIMATED) {
                    put_be32(p + 8, n_frames);
                    put_be32(p + 12, 0u);  // num_plays 0: loop for ever
                    write_chunk(p, "acTL", 8, s_table);
                    p += ACTL_BYTES;
                }
            }
            if constexpr (ANIMATED) {
                put_be32(p + 8, fctl_seq);
                put_be32(p + 12, width);
                put_be32(p + 16, height);
                put_be32(p + 20, 0u);  // x and y offsets: every frame is full size
                put_be32(p + 24, 0u);
                put_be32(p + 28, delay);
                p[32] = 0, p[33] = 0;  // dispose_op NONE, blend_op SOURCE
                write_chunk(p, "fcTL", 26, s_table);
                p += FCTL_BYTES;
            }
            if (first) {
                p[8] = 0x78, p[9] = 0x01;
                write_chunk(p, "IDAT", 2, s_table);
            } else {
                put_be32(p + 8, fctl_seq + 1u);
                p[12] = 0x78, p[13] = 0x01;
                write_chunk(p, "fdAT", 6, s_table);
            }
        }
        return;
    }
    const uint32_t adler = adler_of_rows(sc, width, height, s_red, s_red2);
    if (threadIdx.x == 0) {
        uint8_t *last = out + off, *d = last + 8 + seq_bytes;
        if (!first) put_be32(last + 8, fctl_seq + bands + 2u);
        d[0] = 0x03, d[1] = 0x00;  // BFINAL 1, BTYPE 01, end-of-block
        put_be32(d + 2, adler);
        write_chunk(last, first ? "IDAT" : "fdAT", 6 + seq_bytes, s_table);
        unsigned long long end = off + 18 + seq_bytes;
        if (!ANIMATED || frame + 1u == n_frames) write_chunk(out + end, "IEND", 0, s_table), end += 12;
        *len_word = end;
    }
}

__global__ void __launch_bounds__(WARPS * 32) png_assemble(uint32_t width, uint32_t height, Scratch sc,
                                                             uint8_t *__restrict__ out, unsigned long long *len_word) {
    assemble<false>(width, height, sc, 0, 1, 0, out, len_word);
}

__global__ void __launch_bounds__(WARPS * 32) apng_assemble(uint32_t width, uint32_t height, Scratch sc,
                                                              uint32_t frame, uint32_t n_frames, uint32_t delay,
                                                              uint8_t *__restrict__ out, unsigned long long *len_word) {
    assemble<true>(width, height, sc, frame, n_frames, delay, out, len_word);
}

// The scratch block's pieces (rt_png_scratch_bytes) for a frame of layout `l`.
Scratch scratch_at(const Layout &l, void *scratch) {
    uint8_t *p = static_cast<uint8_t *>(scratch);
    Scratch sc;
    sc.stage = reinterpret_cast<uint32_t *>(p);
    sc.masks = reinterpret_cast<uint32_t *>(p + l.stage_bytes);
    sc.rows = reinterpret_cast<uint4 *>(p + l.stage_bytes + l.mask_bytes);
    sc.bands = reinterpret_cast<uint2 *>(p + l.stage_bytes + l.mask_bytes + l.rows_bytes);
    sc.slot_words = l.slot_words;
    sc.mask_stride = l.mask_stride;
    return sc;
}

}  // namespace

size_t rt_png_bound_bytes(uint32_t width, uint32_t height, const Animation *anim) {
    const Layout l = layout_of(width, height);
    const size_t piece = (3 + 9ull * l.n + 10 + 7) / 8 + 4;
    const size_t png = HEADER_BYTES + 12ull * l.bands + (size_t)height * piece + TRAILER_BYTES;
    return anim ? png + ACTL_BYTES + FCTL_BYTES + 4ull * (l.bands + 2) : png;
}

size_t rt_png_scratch_bytes(uint32_t width, uint32_t height) {
    const Layout l = layout_of(width, height);
    return l.stage_bytes + l.mask_bytes + l.rows_bytes + l.bands_bytes;
}

cudaError_t rt_launch_png_encode(const uint8_t *rgba, size_t pitch, uint32_t width, uint32_t height, const Animation *anim,
                                 uint32_t frame, void *scratch, uint8_t *out, unsigned long long *len_word,
                                 cudaStream_t stream) {
    if (width == 0 || height == 0 || (anim && frame >= anim->n_frames)) return cudaErrorInvalidValue;
    const Layout l = layout_of(width, height);
    const Scratch sc = scratch_at(l, scratch);
    png_encode_rows<<<l.bands, WARPS * 32, 0, stream>>>(rgba, pitch, width, height, sc);
    if (anim)
        apng_assemble<<<l.bands + 1, WARPS * 32, 0, stream>>>(width, height, sc, frame, anim->n_frames,
                                                              (uint32_t)anim->delay_num << 16 | anim->delay_den, out,
                                                              len_word);
    else
        png_assemble<<<l.bands + 1, WARPS * 32, 0, stream>>>(width, height, sc, out, len_word);
    return cudaGetLastError();
}
