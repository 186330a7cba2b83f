// rt_exr.cu -- OpenEXR files encoded on the device (rt_encode_exr).
//
// The layout is fixed so that there is exactly one byte string per image (tests/_exr_ref.py is the reference
// encoder; DESIGN.md "OpenEXR output" explains the choices):
//   single-part scanline OpenEXR, version 2, flags 0; header attributes channels, compression (ZIP), dataWindow,
//   displayWindow, lineOrder (increasing Y), pixelAspectRatio, screenWindowCenter, screenWindowWidth; every channel
//   FLOAT, sampling 1 1, listed in byte order of the name: A B G R, and with the AOV frame also Z coverage.Y
//   normal.X normal.Y normal.Z position.X position.Y position.Z; the offset table; one chunk per 16 scanlines,
//   int32 y0, int32 size, data.
// A chunk's uncompressed bytes are, per scanline and channel, W little-endian floats.  ZIP splits them into even
// then odd bytes and predicts d[i] = t[i] - t[i-1] + 128 (mod 256); its data is one zlib stream of d, or the
// uncompressed bytes when that stream would not be smaller.  The stream is "78 01", pieces of d of 16 KiB framed as
// in rt_deflate.cuh, "03 00" and the Adler-32.  Parse rule of a piece (indices chunk-global, runs inside the piece):
//   far[i]  = D2 && i >= D2 && d[i] == d[i-D2], D2 = 2W when 2W <= 32768 (the same pixel's byte in the previous
//             channel) and no D2 otherwise; a far run is a maximal run of far bytes of length >= 3;
//   near[i] = i >= 1 && d[i] == d[i-1] && i is in no far run; a near run is a maximal run of near bytes;
//   a run of R bytes is floor(R/258) matches of 258, then one match of R mod 258 if that is >= 3, else R mod 258
//   literals; far matches have distance D2, near ones distance 1; every other byte is a literal.
//
// Two launches: exr_encode_pieces (one warp per piece: the far and near masks in shared memory, token bit offsets by
// warp scans, bits packed in shared memory and flushed to the piece's staging slot, the piece's Adler-32 partials),
// then exr_assemble (one CTA per chunk: the chunk's place from the sizes of the chunks before it, compressed or raw,
// its pieces or its raw bytes copied into the file; CTA 0 also writes the header, the last CTA the length).
#include "rt_exr.h"
#include "rt_deflate.cuh"

namespace {

constexpr uint32_t LINES = 16;                 // scanlines per chunk (OpenEXR's ZIP compression)
constexpr uint32_t PIECE = 16384;              // predicted bytes per piece
constexpr uint32_t PIECE_WORDS = PIECE / 32;   // mask words of a piece
constexpr uint32_t WARPS = 8;                  // warps of a CTA (pieces of exr_encode_pieces)
constexpr uint32_t SLOT_WORDS = ((3 + 9 * PIECE + 31) / 32 + 31) / 32 * 32;  // 9 bits per byte at most
constexpr uint32_t MAX_CHANNELS = 12;
// Source of channel k (in name order) as nibble k: 0-3 a float of the colour pixel {r, g, b, alpha}, 8-15 float
// (v - 8) of the AOV pixel {nx, ny, nz, coverage, distance, px, py, pz}.  Nibbles from the lowest: A=3 B=2 G=1 R=0,
// Z=8+4, coverage.Y=8+3, normal.X/Y/Z=8+0/1/2, position.X/Y/Z=8+5/6/7.
constexpr unsigned long long SOURCES = 0xFEDA98BC0123ull;

__host__ __device__ const char *channel_name(uint32_t k) {
    switch (k) {
    case 0: return "A";
    case 1: return "B";
    case 2: return "G";
    case 3: return "R";
    case 4: return "Z";
    case 5: return "coverage.Y";
    case 6: return "normal.X";
    case 7: return "normal.Y";
    case 8: return "normal.Z";
    case 9: return "position.X";
    case 10: return "position.Y";
    default: return "position.Z";
    }
}

__host__ __device__ uint32_t str_len(const char *s) {
    uint32_t n = 0;
    while (s[n]) n++;
    return n;
}

// Bytes of the header (magic, version, the attributes, the terminating 0) of a file of `channels` channels.
uint32_t header_bytes(uint32_t channels) {
    uint32_t chlist = 1;
    for (uint32_t k = 0; k < channels; k++) chlist += str_len(channel_name(k)) + 1 + 16;
    const uint32_t attr = 4;  // each attribute: name\0 type\0 int32 size, then the value
    return 8 + (9 + 7 + attr + chlist) + (12 + 12 + attr + 1) + (11 + 6 + attr + 16) + (14 + 6 + attr + 16) +
           (10 + 10 + attr + 1) + (17 + 6 + attr + 4) + (19 + 4 + attr + 8) + (18 + 6 + attr + 4) + 1;
}

struct Geo {
    const uint8_t *rgba, *aov;         // the frames (aov: null for a colour-only file)
    size_t rgba_pitch, aov_pitch;      // bytes per row
    uint32_t width, height, channels;  // channels: 4 or 12
    uint32_t w4, line;                 // bytes of one channel of a scanline (4W), of a scanline (channels * 4W)
    uint32_t chunks, ppc;              // chunks, pieces of a full chunk (the last chunk may have fewer)
    uint32_t d2, far_dist, far_bits;   // D2 (0: none), its distance code + extra bits (LSB-first) and their length
    uint32_t header;                   // header bytes
    uint32_t *stage;                   // per piece: SLOT_WORDS words of token bits (LSB-first)
    uint4 *rec;                        // per piece: {bits, sum of bytes mod 65521, weighted sum mod 65521, 0}
};

__device__ __forceinline__ uint32_t chunk_bytes(const Geo &g, uint32_t c) { return min(LINES, g.height - c * LINES) * g.line; }

// Where an uncompressed byte lives: image row, channel (name order), byte within the channel's 4W bytes of the row.
struct Cur {
    uint32_t y, ch, off;
};

// Byte b of the uncompressed bytes of the chunk starting at row y0.
__device__ __forceinline__ Cur cur_of_raw(const Geo &g, uint32_t y0, uint32_t b) {
    Cur c;
    const uint32_t s = b / g.line, r = b - s * g.line;
    c.y = y0 + s;
    c.ch = r / g.w4;
    c.off = r - c.ch * g.w4;
    return c;
}

// Predicted byte i of a chunk of n bytes: t[i] is uncompressed byte 2i below the split point n/2, else 2(i - n/2) + 1.
__device__ __forceinline__ Cur cur_of(const Geo &g, uint32_t y0, uint32_t n, uint32_t i) {
    const uint32_t half = n / 2;
    return cur_of_raw(g, y0, i < half ? 2u * i : 2u * (i - half) + 1u);
}

// `bytes` uncompressed bytes further on.
__device__ __forceinline__ void advance(const Geo &g, Cur &c, uint32_t bytes) {
    c.off += bytes;
    while (c.off >= g.w4) {
        c.off -= g.w4;
        if (++c.ch == g.channels) c.ch = 0, c.y++;
    }
}

// The same byte of the same pixel in the channel before (4W uncompressed bytes back).
__device__ __forceinline__ Cur prev_channel(const Geo &g, Cur c) {
    if (c.ch == 0) c.ch = g.channels, c.y--;
    c.ch--;
    return c;
}

__device__ __forceinline__ uint32_t byte_at(const Geo &g, const Cur &c) {
    const uint32_t src = (uint32_t)(SOURCES >> (4u * c.ch)) & 15u, x = c.off >> 2, k = c.off & 3u;
    const uint8_t *p = src < 8u ? g.rgba + c.y * g.rgba_pitch + 16u * x + 4u * src
                                : g.aov + c.y * g.aov_pitch + 32u * x + 4u * (src - 8u);
    return __ldg(p + k);
}

__device__ __forceinline__ uint32_t t_at(const Geo &g, uint32_t y0, uint32_t n, uint32_t i) {
    return byte_at(g, cur_of(g, y0, n, i));
}

__device__ __forceinline__ uint32_t d_at(const Geo &g, uint32_t y0, uint32_t n, uint32_t i) {
    const uint32_t t = t_at(g, y0, n, i);
    return i ? (t - t_at(g, y0, n, i - 1u) + 128u) & 255u : t;
}

// The predicted bytes of a piece, 32 per step (lane = byte): the cursor of this lane's byte and the byte before
// lane 0's.
struct Walk {
    Cur cu;
    bool odd;          // the cursor is in the odd half
    uint32_t carry_t;  // t[i - 1] of lane 0's byte i
};

__device__ __forceinline__ Walk walk_start(const Geo &g, uint32_t y0, uint32_t n, uint32_t i0, uint32_t lane) {
    Walk w;
    w.cu = cur_of(g, y0, n, i0 + lane);
    w.odd = i0 + lane >= n / 2;
    w.carry_t = i0 ? t_at(g, y0, n, i0 - 1u) : 0u;
    return w;
}

// Step k's byte i of this lane: t[i] (0 past the piece) and d[i].
__device__ __forceinline__ void walk_step(const Geo &g, uint32_t y0, uint32_t n, Walk &w, uint32_t k, uint32_t i,
                                          bool valid, uint32_t lane, uint32_t *t, uint32_t *d) {
    if (k) {
        if (!w.odd && i >= n / 2) w.cu = cur_of(g, y0, n, i), w.odd = true;
        else advance(g, w.cu, 64u);
    }
    const uint32_t tv = valid ? byte_at(g, w.cu) : 0u;
    const uint32_t up = __shfl_up_sync(FULL, tv, 1);
    const uint32_t tp = lane ? up : w.carry_t;
    *t = tv;
    *d = i ? (tv - tp + 128u) & 255u : tv;
    w.carry_t = __shfl_sync(FULL, tv, 31);
}

// One warp per piece.  Piece j of chunk c covers predicted bytes [j * PIECE, min(n, (j + 1) * PIECE)).
__global__ void __launch_bounds__(WARPS * 32) exr_encode_pieces(const Geo g) {
    __shared__ uint32_t s_far[WARPS][PIECE_WORDS], s_near[WARPS][PIECE_WORDS];  // run masks, bit p = piece byte p
    __shared__ uint32_t s_buf[WARPS][64];                                      // a warp's pending output words
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t piece = blockIdx.x * WARPS + warp, c = piece / g.ppc, j = piece - c * g.ppc;
    if (c >= g.chunks) return;
    const uint32_t y0 = c * LINES, n = chunk_bytes(g, c), i0 = j * PIECE;
    if (i0 >= n) return;  // the last chunk has fewer pieces
    const uint32_t len = min(PIECE, n - i0), nw = (len + 31u) / 32u;
    uint32_t *fm = s_far[warp], *nm = s_near[warp], *buf = s_buf[warp];
    const uint32_t d2 = g.d2;

    // pass 1: which bytes equal the byte D2 before (far) and the byte before (near)
    {
        Walk w = walk_start(g, y0, n, i0, lane);
        uint32_t carry_d = i0 ? d_at(g, y0, n, i0 - 1u) : 0u;                     // d[i - 1] of lane 0
        uint32_t carry_f = d2 && i0 >= d2 + 1u ? t_at(g, y0, n, i0 - d2 - 1u) : 0u;  // t[i - D2 - 1] of lane 0
        for (uint32_t k = 0; k < nw; k++) {
            const uint32_t p = k * 32u + lane, i = i0 + p;
            const bool valid = p < len;
            uint32_t tv, dv;
            walk_step(g, y0, n, w, k, i, valid, lane, &tv, &dv);
            const bool fok = valid && d2 && i >= d2;
            uint32_t tf = 0;
            if (fok) tf = byte_at(g, (!w.odd || i - d2 >= n / 2) ? prev_channel(g, w.cu) : cur_of(g, y0, n, i - d2));
            const uint32_t upf = __shfl_up_sync(FULL, tf, 1), upd = __shfl_up_sync(FULL, dv, 1);
            const uint32_t tfp = lane ? upf : carry_f, dp = lane ? upd : carry_d;
            const uint32_t df = i - d2 ? (tf - tfp + 128u) & 255u : tf;
            const uint32_t f = __ballot_sync(FULL, fok && df == dv);
            const uint32_t e = __ballot_sync(FULL, valid && i >= 1u && dv == dp);
            if (lane == 0) fm[k] = f, nm[k] = e;
            carry_f = __shfl_sync(FULL, tf, 31);
            carry_d = __shfl_sync(FULL, dv, 31);
        }
        __syncwarp();
        // far runs: far bytes in a run of >= 3 (bit i of `tri` = bytes i, i+1, i+2 are far); near: not in a far run
        uint32_t runs[PIECE_WORDS / 32];
#pragma unroll
        for (uint32_t m = 0; m < PIECE_WORDS / 32; m++) {
            const uint32_t k = m * 32u + lane;
            runs[m] = 0;
            if (k < nw) {
                const uint32_t f0 = k ? fm[k - 1] : 0u, f1 = fm[k], f2 = k + 1u < nw ? fm[k + 1] : 0u;
                const uint32_t t0 = f0 & (f0 >> 1 | f1 << 31) & (f0 >> 2 | f1 << 30);
                const uint32_t t1 = f1 & (f1 >> 1 | f2 << 31) & (f1 >> 2 | f2 << 30);
                runs[m] = t1 | (t1 << 1 | t0 >> 31) | (t1 << 2 | t0 >> 30);
            }
        }
        __syncwarp();
#pragma unroll
        for (uint32_t m = 0; m < PIECE_WORDS / 32; m++) {
            const uint32_t k = m * 32u + lane;
            if (k < nw) fm[k] = runs[m], nm[k] &= ~runs[m];
        }
        buf[lane] = lane == 0 ? 2u : 0u;  // the piece's block header: BFINAL 0, BTYPE 01 is bit value 2
        buf[lane + 32] = 0;
        __syncwarp();
    }

    // pass 2: token bit offsets (a run's matches are charged to its first byte, its trailing literals to themselves,
    // so an exclusive scan gives every token's offset), the tokens, the Adler-32 partials
    const uint32_t sym285 = __brev(0xC5u) >> 24;
    const uint32_t far258 = sym285 | g.far_dist << 8, far258_bits = 8u + g.far_bits;  // near: distance 1 is code 0
    uint32_t *stage = g.stage + (size_t)piece * SLOT_WORDS;
    Walk w = walk_start(g, y0, n, i0, lane);
    uint32_t bits = 3, base_word = 0;
    uint32_t run_s = 0, run_len = 0, run_off = 0;  // the run reaching into this step from earlier ones
    bool run_far = false;
    uint32_t prev_f = 0, prev_n = 0;
    unsigned long long sum = 0, wsum = 0;
    for (uint32_t k = 0; k < nw; k++) {
        const uint32_t p = k * 32u + lane, i = i0 + p;
        const bool valid = p < len;
        uint32_t tv, v;
        walk_step(g, y0, n, w, k, i, valid, lane, &tv, &v);
        const uint32_t mf = fm[k], mn = nm[k];
        const bool is_f = (mf >> lane) & 1u, is_n = (mn >> lane) & 1u, member = is_f || is_n;
        const bool pf = lane ? (mf >> (lane - 1u)) & 1u : prev_f, pn = lane ? (mn >> (lane - 1u)) & 1u : prev_n;
        const bool start = (is_f && !pf) || (is_n && !pn);
        uint32_t R = 0;
        if (start) {  // the run ends at the first clear bit of its mask at or after p (bits past the piece are clear)
            const uint32_t *mask = is_f ? fm : nm;
            uint32_t wk = k, z = ~mask[k] & (FULL << lane);
            while (z == 0 && ++wk < nw) z = ~mask[wk];
            const uint32_t t = z ? min(wk * 32u + __ffs(z) - 1u, len) : len;
            R = t - p;
        }
        // the run this byte belongs to: the highest run start at or below this lane, else the carried one
        const uint32_t starts = __ballot_sync(FULL, start);
        const uint32_t le = starts & (FULL >> (31u - lane));
        const int src = le ? 31 - __clz(le) : (int)lane;
        const uint32_t ss = __shfl_sync(FULL, p, src), sR = __shfl_sync(FULL, R, src);
        const bool sf = __shfl_sync(FULL, (uint32_t)is_f, src);
        const uint32_t rs = le ? ss : run_s, rl = le ? sR : run_len;
        const bool rf = le ? sf : run_far;
        const uint32_t j = p - rs, q = rl / 258u, tail = 258u * q, rr = rl - tail;
        const uint32_t m_bits = rf ? far258_bits : 13u, m_dist = rf ? g.far_dist : 0u, m_dbits = rf ? g.far_bits : 5u;
        const bool literal = valid && (!member || (j >= tail && rr < 3u));
        uint32_t cost = literal ? lit_bits(v) : 0u;
        if (start) {
            cost += m_bits * q;
            if (rr >= 3u) {
                uint32_t nb;
                match_code(rr, m_dist, m_dbits, &nb);
                cost += nb;
            }
        }
        uint32_t inc = cost;
#pragma unroll
        for (uint32_t dd = 1; dd < 32; dd <<= 1) {
            const uint32_t o = __shfl_up_sync(FULL, inc, dd);
            if (lane >= dd) inc += o;
        }
        const uint32_t off = bits + inc - cost;
        const uint32_t so = __shfl_sync(FULL, off, src);
        const uint32_t ro = le ? so : run_off;
        uint32_t code = 0, nb = 0, o = 0;
        if (literal) {
            code = lit_code(v), nb = lit_bits(v), o = off;  // a start that is a literal has no match before it
        } else if (member) {
            if (j < tail) {
                if (j % 258u == 0) code = rf ? far258 : sym285, nb = m_bits, o = ro + m_bits * (j / 258u);
            } else if (j == tail) {
                code = match_code(rr, m_dist, m_dbits, &nb), o = ro + m_bits * q;
            }
        }
        if (nb) {
            const uint32_t wd = (o >> 5) - base_word, sh = o & 31u;
            atomicOr(&buf[wd], code << sh);
            if (sh + nb > 32u) atomicOr(&buf[wd + 1], code >> (32u - sh));
        }
        if (valid) sum += v, wsum += (unsigned long long)(len - p) * v;
        bits += __shfl_sync(FULL, inc, 31);
        if (starts) {
            const int hi = 31 - __clz(starts);
            run_s = __shfl_sync(FULL, p, hi), run_len = __shfl_sync(FULL, R, hi), run_off = __shfl_sync(FULL, off, hi);
            run_far = __shfl_sync(FULL, (uint32_t)is_f, hi);
        }
        prev_f = mf >> 31, prev_n = mn >> 31;
        // bits below `frontier` are final: everything, unless a run continues into the next step -- then up to the
        // token covering this step's last byte
        const uint32_t last = k * 32u + 31u;
        const uint32_t frontier = ((prev_f | prev_n) && run_s + run_len > last + 1u)
                                      ? run_off + (run_far ? far258_bits : 13u) * ((last - run_s) / 258u)
                                      : bits;
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
    for (uint32_t q = lane; base_word + q < words; q += 32u) stage[base_word + q] = buf[q];
    for (uint32_t dd = 16; dd; dd >>= 1) {
        sum += __shfl_xor_sync(FULL, sum, dd);
        wsum += __shfl_xor_sync(FULL, wsum, dd);
    }
    if (lane == 0) g.rec[piece] = make_uint4(bits, (uint32_t)(sum % ADLER_MOD), (uint32_t)(wsum % ADLER_MOD), 0u);
}

// ---- exr_assemble -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pieces_of(uint32_t n) { return (n + PIECE - 1u) / PIECE; }

// The zlib stream of chunk c (warp-wide; every lane gets it): "78 01", the pieces, "03 00", the Adler-32.
__device__ uint32_t zlib_bytes(const Geo &g, uint32_t c, uint32_t lane) {
    const uint32_t np = pieces_of(chunk_bytes(g, c));
    uint32_t s = 0;
    for (uint32_t j = lane; j < np; j += 32u) s += piece_bytes(g.rec[c * g.ppc + j].x);
    for (uint32_t dd = 16; dd; dd >>= 1) s += __shfl_xor_sync(FULL, s, dd);
    return 2u + s + 6u;
}

// The data of chunk c: its zlib stream if that is smaller than its uncompressed bytes, else those bytes.
__device__ __forceinline__ uint32_t data_bytes(const Geo &g, uint32_t c, uint32_t lane) {
    return min(zlib_bytes(g, c, lane), chunk_bytes(g, c));
}

__device__ __forceinline__ uint8_t *put_u32(uint8_t *p, uint32_t v) {
    for (int k = 0; k < 4; k++) p[k] = (uint8_t)(v >> (8 * k));
    return p + 4;
}

__device__ uint8_t *put_attr(uint8_t *p, const char *name, const char *type, uint32_t size) {
    for (const char *s = name; *s; s++) *p++ = (uint8_t)*s;
    *p++ = 0;
    for (const char *s = type; *s; s++) *p++ = (uint8_t)*s;
    *p++ = 0;
    return put_u32(p, size);
}

__device__ void write_header(const Geo &g, uint8_t *p) {
    p = put_u32(p, 20000630u);  // magic 76 2f 31 01
    p = put_u32(p, 2u);         // version 2, single-part scanline, no flags
    uint32_t chlist = 1;
    for (uint32_t k = 0; k < g.channels; k++) chlist += str_len(channel_name(k)) + 1u + 16u;
    p = put_attr(p, "channels", "chlist", chlist);
    for (uint32_t k = 0; k < g.channels; k++) {
        for (const char *s = channel_name(k); *s; s++) *p++ = (uint8_t)*s;
        *p++ = 0;
        p = put_u32(p, 2u);  // FLOAT
        p = put_u32(p, 0u);  // pLinear 0, reserved
        p = put_u32(p, 1u);  // xSampling
        p = put_u32(p, 1u);  // ySampling
    }
    *p++ = 0;
    p = put_attr(p, "compression", "compression", 1);
    *p++ = 3;  // ZIP_COMPRESSION: 16 scanlines per chunk
    for (int k = 0; k < 2; k++) {
        p = put_attr(p, k ? "displayWindow" : "dataWindow", "box2i", 16);
        p = put_u32(p, 0u), p = put_u32(p, 0u), p = put_u32(p, g.width - 1u), p = put_u32(p, g.height - 1u);
    }
    p = put_attr(p, "lineOrder", "lineOrder", 1);
    *p++ = 0;  // INCREASING_Y
    p = put_attr(p, "pixelAspectRatio", "float", 4);
    p = put_u32(p, 0x3f800000u);
    p = put_attr(p, "screenWindowCenter", "v2f", 8);
    p = put_u32(p, 0u), p = put_u32(p, 0u);
    p = put_attr(p, "screenWindowWidth", "float", 4);
    p = put_u32(p, 0x3f800000u);
    *p = 0;
}

// One CTA per chunk: its place in the file, its offset-table entry, y0 and size, then its zlib stream (the pieces
// back to back between "78 01" and "03 00" + Adler-32) or its uncompressed bytes.  CTA 0 also writes the header, the
// last CTA the file's length.
__global__ void __launch_bounds__(WARPS * 32) exr_assemble(const Geo g, uint8_t *__restrict__ out,
                                                           unsigned long long *len_word) {
    __shared__ unsigned long long s_red[WARPS], s_red2[WARPS];
    __shared__ uint32_t s_size;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, c = blockIdx.x;
    const uint32_t n = chunk_bytes(g, c), np = pieces_of(n), p0 = c * g.ppc;
    unsigned long long acc = 0;
    for (uint32_t cc = warp; cc < c; cc += WARPS) acc += 8u + data_bytes(g, cc, lane);
    if (lane == 0) s_red[warp] = acc;
    if (warp == 0) {
        const uint32_t z = zlib_bytes(g, c, lane);
        if (lane == 0) s_size = z;
    }
    __syncthreads();
    unsigned long long off = g.header + 8ull * g.chunks;
    for (uint32_t w = 0; w < WARPS; w++) off += s_red[w];
    const uint32_t zsize = s_size, size = min(zsize, n);
    uint8_t *data = out + off + 8;
    if (threadIdx.x == 0) {
        uint8_t *t = out + g.header + 8ull * c;
        put_u32(t, (uint32_t)off), put_u32(t + 4, (uint32_t)(off >> 32));
        put_u32(out + off, c * LINES);
        put_u32(out + off + 4, size);
        if (c == 0) write_header(g, out);
        if (c + 1u == g.chunks) *len_word = off + 8u + size;
    }
    if (size == n) {  // raw: the uncompressed bytes, one float per thread and step
        const uint32_t floats = n / 4u, per_line = g.channels * g.width;
        for (uint32_t f = threadIdx.x; f < floats; f += blockDim.x) {
            const uint32_t s = f / per_line, r = f - s * per_line, ch = r / g.width, x = r - ch * g.width;
            Cur cu;
            cu.y = c * LINES + s, cu.ch = ch, cu.off = 4u * x;
            uint8_t *d = data + 4u * f;
            for (uint32_t k = 0; k < 4; k++, cu.off++) d[k] = (uint8_t)byte_at(g, cu);
        }
        return;
    }
    // the pieces, warp w taking pieces w, w + WARPS, ...; `pre` is the offset of piece j in the stream
    uint32_t pre = 2, done = 0;
    for (uint32_t j = warp; j < np; j += WARPS) {
        uint32_t part = 0;
        for (uint32_t jj = done + lane; jj < j; jj += 32u) part += piece_bytes(g.rec[p0 + jj].x);
        for (uint32_t dd = 16; dd; dd >>= 1) part += __shfl_xor_sync(FULL, part, dd);
        pre += part, done = j;
        const uint32_t bits = g.rec[p0 + j].x, len = piece_bytes(bits);
        const uint8_t *staged = reinterpret_cast<const uint8_t *>(g.stage + (size_t)(p0 + j) * SLOT_WORDS);
        uint8_t *d = data + pre;
        for (uint32_t q = lane; q < len; q += 32u) d[q] = (uint8_t)piece_byte(staged, bits, len, q);
    }
    // the Adler-32 of the predicted bytes from the per-piece partials: piece j of L_j bytes starts at byte a_j of n,
    // so b gains W_j + (n - a_j - L_j) * S_j, where S_j = sum of its bytes and W_j = sum of (L_j - k) * byte k
    unsigned long long sa = 0, sb = 0;
    for (uint32_t j = threadIdx.x; j < np; j += blockDim.x) {
        const uint4 r = g.rec[p0 + j];
        const uint32_t a = j * PIECE, l = min(PIECE, n - a);
        sa += r.y;
        sb += (r.z + (unsigned long long)((n - a - l) % ADLER_MOD) * r.y) % ADLER_MOD;
    }
    for (uint32_t dd = 16; dd; dd >>= 1) sa += __shfl_xor_sync(FULL, sa, dd), sb += __shfl_xor_sync(FULL, sb, dd);
    __syncthreads();  // s_red is reused
    if (lane == 0) s_red[warp] = sa, s_red2[warp] = sb;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long a = 1, b = n % ADLER_MOD;
        for (uint32_t w = 0; w < WARPS; w++) a += s_red[w], b += s_red2[w];
        a %= ADLER_MOD, b %= ADLER_MOD;
        data[0] = 0x78, data[1] = 0x01;
        uint8_t *e = data + zsize - 6u;
        e[0] = 0x03, e[1] = 0x00;  // BFINAL 1, BTYPE 01, end-of-block
        e[2] = (uint8_t)(b >> 8), e[3] = (uint8_t)b, e[4] = (uint8_t)(a >> 8), e[5] = (uint8_t)a;
    }
}

Geo geo_of(uint32_t width, uint32_t height, bool aov) {
    Geo g{};
    g.width = width, g.height = height, g.channels = aov ? MAX_CHANNELS : 4u;
    g.w4 = 4u * width, g.line = g.channels * g.w4;
    g.chunks = (height + LINES - 1) / LINES;
    g.ppc = (min(LINES, height) * g.line + PIECE - 1) / PIECE;
    g.d2 = 2u * width <= 32768u ? 2u * width : 0u;
    if (g.d2) {  // RFC 1951 3.2.5: distance code and extra bits of D2
        const uint32_t d = g.d2 - 1u;
        uint32_t code = d, extra = 0, ebits = 0;
        if (g.d2 > 4u) {
            const uint32_t top = 31u - (uint32_t)__builtin_clz(d);
            ebits = top - 1u;
            code = 2u * top + ((d >> ebits) & 1u);
            extra = d & ((1u << ebits) - 1u);
        }
        uint32_t rev = 0;
        for (int k = 0; k < 5; k++) rev |= ((code >> k) & 1u) << (4 - k);
        g.far_dist = rev | extra << 5;
        g.far_bits = 5u + ebits;
    }
    g.header = header_bytes(g.channels);
    return g;
}

size_t stage_bytes(const Geo &g) { return (size_t)g.chunks * g.ppc * SLOT_WORDS * 4; }

}  // namespace

size_t rt_exr_bound_bytes(uint32_t width, uint32_t height, bool aov) {
    const Geo g = geo_of(width, height, aov);
    return g.header + 16ull * g.chunks + (size_t)height * g.line;
}

size_t rt_exr_scratch_bytes(uint32_t width, uint32_t height, bool aov) {
    const Geo g = geo_of(width, height, aov);
    return stage_bytes(g) + (size_t)g.chunks * g.ppc * sizeof(uint4);
}

cudaError_t rt_launch_exr_encode(const float *rgba, size_t rgba_pitch, const float *aov, size_t aov_pitch,
                                 uint32_t width, uint32_t height, void *scratch, uint8_t *out,
                                 unsigned long long *len_word, cudaStream_t stream) {
    if (width == 0 || height == 0 || !rgba) return cudaErrorInvalidValue;
    Geo g = geo_of(width, height, aov != nullptr);
    g.rgba = reinterpret_cast<const uint8_t *>(rgba), g.rgba_pitch = rgba_pitch;
    g.aov = reinterpret_cast<const uint8_t *>(aov), g.aov_pitch = aov_pitch;
    g.stage = static_cast<uint32_t *>(scratch);
    g.rec = reinterpret_cast<uint4 *>(static_cast<uint8_t *>(scratch) + stage_bytes(g));
    const uint32_t pieces = g.chunks * g.ppc;
    exr_encode_pieces<<<(pieces + WARPS - 1) / WARPS, WARPS * 32, 0, stream>>>(g);
    exr_assemble<<<g.chunks, WARPS * 32, 0, stream>>>(g, out, len_word);
    return cudaGetLastError();
}
