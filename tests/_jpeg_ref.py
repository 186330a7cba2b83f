"""Reference encoder of rt_encode_jpeg's JPEG layout (DESIGN.md "JPEG output"), in numpy.

The file is baseline sequential JPEG, 4:2:0, the standard Huffman tables of ITU T.81 Annex K, and one restart interval
per MCU row: the bytes libjpeg(-turbo) writes for `Image.fromarray(rgb).save(f, "JPEG", quality=q, subsampling=2,
restart_marker_rows=1)`.  Every step is libjpeg's integer arithmetic (jcparam.c, jccolor.c, jcsample.c, jcprepct.c,
jccoefct.c, jfdctint.c, jcdctmgr.c, jchuff.c, jcmarker.c), restated over whole frames at once so that a 4K frame takes
seconds.  Nothing here uses Pillow; the tests compare it with Pillow's bytes.
"""
import numpy as np

# ITU T.81 Annex K: the example quantisation tables (natural order) and Huffman tables (BITS, HUFFVAL)
BASE_QUANT = (
    np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
              14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
              49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99], dtype=np.int64),
    np.array([17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
              47, 66, 99, 99, 99, 99, 99, 99] + [99] * 32, dtype=np.int64),
)
# (BITS[1..16], HUFFVAL) of DC luma, AC luma, DC chroma, AC chroma, in the order the DHT markers carry them
HUFF = {
    "dc0": ("00010501010101010100000000000000", "000102030405060708090a0b"),
    "ac0": ("0002010303020403050504040000017d",
            "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a"
            "3435363738393a434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a929394"
            "95969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8"
            "e9eaf1f2f3f4f5f6f7f8f9fa"),
    "dc1": ("00030101010101010101010000000000", "000102030405060708090a0b"),
    "ac1": ("00020102040403040705040400010277",
            "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728"
            "292a35363738393a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92"
            "939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7"
            "e8e9eaf2f3f4f5f6f7f8f9fa"),
}

# zig-zag position -> natural (row-major) index
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20,
                   13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52,
                   45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63], dtype=np.int64)

HEADER_BYTES = 2 + 18 + 2 * 69 + 19 + 2 * 33 + 2 * 183 + 6 + 14  # SOI .. SOS: 629
BLOCK_BITS = 11 + 11 + 63 * (16 + 10)  # the most one 8x8 block can code to (DESIGN.md "JPEG output")


def huff_tables(name):
    """(bits, huffval) and the code/size of every symbol (jchuff.c jpeg_make_c_derived_tbl)."""
    bits = bytes.fromhex(HUFF[name][0])
    vals = bytes.fromhex(HUFF[name][1])
    code = np.zeros(256, np.int64)
    size = np.zeros(256, np.int64)
    c, k = 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            code[vals[k]] = c
            size[vals[k]] = length
            c += 1
            k += 1
        c <<= 1
    return bits, vals, code, size


def quant_tables(quality):
    """Luma and chroma tables (natural order) of jpeg_set_quality(quality, force_baseline=TRUE)."""
    if not 1 <= quality <= 100:
        raise ValueError("quality must be in 1..100")
    scale = 5000 // quality if quality < 50 else 200 - quality * 2
    return tuple(np.clip((b * scale + 50) // 100, 1, 255) for b in BASE_QUANT)


def bound(width, height):
    """rt_jpeg_bound: the header, every MCU row's worst case (every block at BLOCK_BITS, a padding byte, all doubled
    for 0xFF stuffing, plus its RST marker), and EOI."""
    if not (1 <= width <= 65535 and 1 <= height <= 65535):
        raise ValueError("width/height must be in 1..65535")
    mcus = (width + 15) // 16
    rows = (height + 15) // 16
    return HEADER_BYTES + rows * (2 * (mcus * 6 * BLOCK_BITS // 8 + 1) + 2) + 2


def header(width, height, quality):
    """SOI, APP0 JFIF, DQT x2, SOF0, DHT x4, DRI, SOS: the bytes before the first entropy-coded segment."""
    def seg(marker, body):
        return bytes([0xFF, marker]) + (len(body) + 2).to_bytes(2, "big") + body

    q = quant_tables(quality)
    out = b"\xff\xd8" + seg(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for t in (0, 1):
        out += seg(0xDB, bytes([t]) + bytes(int(v) for v in q[t][ZIGZAG]))
    out += seg(0xC0, bytes([8]) + height.to_bytes(2, "big") + width.to_bytes(2, "big")
               + bytes([3, 1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1]))
    for name, tc_th in (("dc0", 0x00), ("ac0", 0x10), ("dc1", 0x01), ("ac1", 0x11)):
        bits, vals, _, _ = huff_tables(name)
        out += seg(0xC4, bytes([tc_th]) + bits + vals)
    out += seg(0xDD, ((width + 15) // 16).to_bytes(2, "big"))
    out += seg(0xDA, bytes([3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0]))
    assert len(out) == HEADER_BYTES
    return out


def ycc(rgb):
    """jccolor.c rgb_ycc_convert: (Y, Cb, Cr) as int64 arrays."""
    r, g, b = (rgb[..., k].astype(np.int64) for k in range(3))
    half, off = 1 << 15, 128 << 16
    y = (19595 * r + 38470 * g + 7471 * b + half) >> 16
    cb = (-11059 * r - 21709 * g + 32768 * b + off + half - 1) >> 16
    cr = (32768 * r - 27439 * g - 5329 * b + off + half - 1) >> 16
    return y, cb, cr


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _fdct_1d(d, axis, final):
    """One pass of jfdctint.c jpeg_fdct_islow along `axis` (length 8) of int64 array d."""
    CB, P1 = 13, 2
    t = [np.take(d, k, axis=axis) for k in range(8)]
    tmp0, tmp7 = t[0] + t[7], t[0] - t[7]
    tmp1, tmp6 = t[1] + t[6], t[1] - t[6]
    tmp2, tmp5 = t[2] + t[5], t[2] - t[5]
    tmp3, tmp4 = t[3] + t[4], t[3] - t[4]
    tmp10, tmp13 = tmp0 + tmp3, tmp0 - tmp3
    tmp11, tmp12 = tmp1 + tmp2, tmp1 - tmp2
    sh = CB + P1 if final else CB - P1
    out = [None] * 8
    if final:
        out[0] = _descale(tmp10 + tmp11, P1)
        out[4] = _descale(tmp10 - tmp11, P1)
    else:
        out[0] = (tmp10 + tmp11) << P1
        out[4] = (tmp10 - tmp11) << P1
    z1 = (tmp12 + tmp13) * 4433
    out[2] = _descale(z1 + tmp13 * 6270, sh)
    out[6] = _descale(z1 - tmp12 * 15137, sh)
    z1, z2, z3, z4 = tmp4 + tmp7, tmp5 + tmp6, tmp4 + tmp6, tmp5 + tmp7
    z5 = (z3 + z4) * 9633
    tmp4, tmp5, tmp6, tmp7 = tmp4 * 2446, tmp5 * 16819, tmp6 * 25172, tmp7 * 12299
    z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
    out[7] = _descale(tmp4 + z1 + z3, sh)
    out[5] = _descale(tmp5 + z2 + z4, sh)
    out[3] = _descale(tmp6 + z2 + z3, sh)
    out[1] = _descale(tmp7 + z1 + z4, sh)
    return np.stack(out, axis=axis)


def fdct_quant(blocks, qtbl):
    """jpeg_fdct_islow of (sample - 128) then jcdctmgr.c quantize (round half away from zero by 8 * qtbl):
    blocks (..., 8, 8) int64 samples -> (..., 64) coefficients in zig-zag order."""
    d = blocks.astype(np.int64) - 128
    d = _fdct_1d(d, -1, False)
    d = _fdct_1d(d, -2, True)
    d = d.reshape(d.shape[:-2] + (64,))
    div = 8 * qtbl
    q = (np.abs(d) + (div >> 1)) // div
    return (np.sign(d) * q)[..., ZIGZAG]


def coefficients(rgb, quality):
    """Quantised coefficients (rows, mcus, 6, 64), zig-zag order, blocks Y00 Y01 Y10 Y11 Cb Cr per MCU."""
    h, w = rgb.shape[:2]
    rows, mcus = (h + 15) // 16, (w + 15) // 16
    # Columns: the last one is replicated out to whole MCUs before downsampling (jcsample.c expand_right_edge), and
    # colour conversion is per pixel, so every column past the image is its last column.  Rows: the image is
    # replicated to an even height, downsampled, and then each component's last row is replicated down to the MCU
    # row (jcprepct.c): luma rows past the image are its last row, chroma rows past (h + 1) / 2 the last chroma row.
    ys = np.minimum(np.arange(rows * 16), h - 1)
    xs = np.minimum(np.arange(mcus * 16), w - 1)
    y, cb, cr = ycc(rgb[ys][:, xs])
    # jcsample.c h2v2_downsample: bias 1, 2, 1, 2, ... along each output row
    bias = np.tile(np.array([1, 2], np.int64), mcus * 4)
    crow = np.minimum(np.arange(rows * 8), (h + 1) // 2 - 1)
    def down(c):
        return ((c[0::2, 0::2] + c[0::2, 1::2] + c[1::2, 0::2] + c[1::2, 1::2] + bias) >> 2)[crow]
    q = quant_tables(quality)
    yb = y.reshape(rows, 2, 8, mcus, 2, 8).transpose(0, 3, 1, 4, 2, 5).reshape(rows, mcus, 4, 8, 8)
    cbb = down(cb).reshape(rows, 8, mcus, 8).transpose(0, 2, 1, 3)[:, :, None]
    crb = down(cr).reshape(rows, 8, mcus, 8).transpose(0, 2, 1, 3)[:, :, None]
    coef = np.concatenate([fdct_quant(yb, q[0]), fdct_quant(cbb, q[1]), fdct_quant(crb, q[1])], axis=2)
    # jccoefct.c dummy blocks: a luma block past the image's last block column or row codes AC zero and the DC of
    # the block before it in the MCU (a bottom dummy: of block Y01, itself possibly a dummy copying Y00)
    wb, hb = (w + 7) // 8, (h + 7) // 8
    if wb % 2:
        coef[:, -1, 1] = 0
        coef[:, -1, 1, 0] = coef[:, -1, 0, 0]
        coef[:, -1, 3] = 0
        coef[:, -1, 3, 0] = coef[:, -1, 2, 0]
    if hb % 2:
        coef[-1, :, 2:4] = 0
        coef[-1, :, 2:4, 0] = coef[-1, :, 1:2, 0]
    return coef


_NBITS = np.array([0] + [int(v).bit_length() for v in range(1, 1 << 12)], dtype=np.int64)


def _pack(values, lengths):
    """Big-endian bit string of the (value, length) items, as bytes; the total length is a multiple of 8."""
    total = int(lengths.sum())
    assert total % 8 == 0
    keep = lengths > 0
    values, lengths = values[keep], lengths[keep]
    starts = np.cumsum(lengths) - lengths
    item = np.repeat(np.arange(len(lengths)), lengths)
    pos = np.arange(total) - starts[item]
    bits = (values[item] >> (lengths[item] - 1 - pos)) & 1
    return np.packbits(bits.astype(np.uint8)).tobytes()


def entropy_segments(coef):
    """One byte string per MCU row: its Huffman-coded blocks (DC predictions reset at the row's start), padded with
    1-bits to a byte, 0xFF bytes stuffed with 0x00."""
    rows, mcus = coef.shape[:2]
    tabs = [huff_tables(n) for n in ("dc0", "ac0", "dc1", "ac1")]
    comp = np.array([0, 0, 0, 0, 1, 1], np.int64)  # 0 luma, 1 chroma, per block of an MCU
    n = rows * mcus * 6
    flat = coef.reshape(n, 64)
    blk_comp = np.tile(comp, rows * mcus)
    blk_row = np.repeat(np.arange(rows), mcus * 6)

    # DC differences, per component, in coding order within a row
    dc = coef[..., 0]
    diff = np.empty_like(dc)
    yd = dc[:, :, :4].reshape(rows, mcus * 4)
    diff[:, :, :4] = np.diff(yd, axis=1, prepend=0).reshape(rows, mcus, 4)
    for b in (4, 5):
        diff[:, :, b] = np.diff(dc[:, :, b], axis=1, prepend=0)
    diff = diff.reshape(n)

    def mag(v, s):  # the s low bits of v, ones' complement for negative v (jchuff.c)
        return np.where(v < 0, v - 1, v) & ((1 << s) - 1)

    keys, vals, lens = [], [], []
    # DC: code of its size category, then the bits
    s = _NBITS[np.abs(diff)]
    dcode = np.where(blk_comp == 0, tabs[0][2][s], tabs[2][2][s])
    dsize = np.where(blk_comp == 0, tabs[0][3][s], tabs[2][3][s])
    keys.append(np.arange(n) * 1024)
    vals.append((dcode << s) | mag(diff, s))
    lens.append(dsize + s)
    # AC: per nonzero coefficient, (run >> 4) ZRL codes, then the code of (run & 15, size) and the bits
    ac = flat[:, 1:]
    bi, zi = np.nonzero(ac)
    z = zi + 1
    v = ac[bi, zi]
    prev = np.zeros_like(z)
    same = np.zeros(len(z), bool)
    same[1:] = bi[1:] == bi[:-1]
    prev[1:] = np.where(same[1:], z[:-1], 0)
    run = z - prev - 1
    s = _NBITS[np.abs(v)]
    sym = ((run & 15) << 4) | s
    luma = blk_comp[bi] == 0
    code = np.where(luma, tabs[1][2][sym], tabs[3][2][sym])
    size = np.where(luma, tabs[1][3][sym], tabs[3][3][sym])
    zrl_code = np.where(luma, tabs[1][2][0xF0], tabs[3][2][0xF0])
    zrl_size = np.where(luma, tabs[1][3][0xF0], tabs[3][3][0xF0])
    for k in range(3):  # a run is at most 62 zeros: at most three ZRL codes
        has = (run >> 4) > k
        keys.append(bi[has] * 1024 + z[has] * 8 + k)
        vals.append(zrl_code[has])
        lens.append(zrl_size[has])
    keys.append(bi * 1024 + z * 8 + 3)
    vals.append((code << s) | mag(v, s))
    lens.append(size + s)
    # EOB where the last coefficient is zero
    last = np.zeros(n, np.int64)
    np.maximum.at(last, bi, z)
    eob = last < 63
    eb = np.nonzero(eob)[0]
    keys.append(eb * 1024 + 1000)
    vals.append(np.where(blk_comp[eb] == 0, tabs[1][2][0], tabs[3][2][0]))
    lens.append(np.where(blk_comp[eb] == 0, tabs[1][3][0], tabs[3][3][0]))

    keys = np.concatenate(keys)
    order = np.argsort(keys, kind="stable")
    vals = np.concatenate(vals)[order]
    lens = np.concatenate(lens)[order]
    row_of = blk_row[keys[order] // 1024]
    # pad every row to a byte with 1-bits: one more item at the end of each row
    row_bits = np.bincount(row_of, weights=lens, minlength=rows).astype(np.int64)
    pad = (-row_bits) % 8
    ends = np.searchsorted(row_of, np.arange(rows), side="right")
    vals = np.insert(vals, ends, (1 << pad) - 1)
    lens = np.insert(lens, ends, pad)
    data = np.frombuffer(_pack(vals, lens), np.uint8)
    cuts = np.cumsum((row_bits + pad) // 8)
    segs = []
    for seg in np.split(data, cuts[:-1]):
        ff = np.nonzero(seg == 0xFF)[0]
        segs.append(np.insert(seg, ff + 1, 0).tobytes())
    return segs


def encode(rgb, quality=90):
    """The JPEG file of an (h, w, 3) or (h, w, 4) uint8 frame (alpha dropped), at `quality` 1..100."""
    rgb = np.ascontiguousarray(rgb[..., :3])
    h, w = rgb.shape[:2]
    bound(w, h)
    segs = entropy_segments(coefficients(rgb, quality))
    out = [header(w, h, quality)]
    for i, seg in enumerate(segs):
        out.append(seg)
        if i + 1 < len(segs):
            out.append(bytes([0xFF, 0xD0 + (i & 7)]))
    out.append(b"\xff\xd9")
    return b"".join(out)
