"""Reference encoder and decoder of the PNG layout rt_encode_png writes.  TEST INFRASTRUCTURE.

The layout (DESIGN.md "PNG output"): 8-bit RGB, colour type 2, no interlace; an IDAT holding the zlib header
78 01; one IDAT per band of 16 image rows, each row one byte-aligned piece (a non-final fixed-Huffman block of
filter byte 0 + the row's RGB bytes, parsed into literals and distance-3 matches by a closed-form rule, then an
empty non-final stored block); a last IDAT holding a final empty fixed block and the Adler-32; IEND.  There is
exactly one byte string per image, so the GPU output is compared with `encode` byte for byte.
"""
import bisect
import struct
import zlib

import numpy as np

LB = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LE = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
BAND = 16
SIGNATURE = b"\x89PNG\r\n\x1a\n"


def rev(c, n):
    return int(format(c, "0%db" % n)[::-1], 2)


def fixed_code(s):                      # RFC 1951 3.2.6, bit-reversed for an LSB-first stream
    if s < 144:
        return rev(0x30 + s, 8), 8
    if s < 256:
        return rev(0x190 + s - 144, 9), 9
    if s < 280:
        return rev(s - 256, 7), 7
    return rev(0xC0 + s - 280, 8), 8


FC = [fixed_code(s) for s in range(288)]


def length_code(L):
    k = bisect.bisect_right(LB, L) - 1
    c, n = FC[257 + k]
    return c | ((L - LB[k]) << n), n + LE[k]


DIST3 = (rev(2, 5), 5)


class Bits:
    def __init__(s):
        s.acc = s.n = 0
        s.out = bytearray()

    def put(s, v, n):
        s.acc |= v << s.n
        s.n += n
        while s.n >= 8:
            s.out.append(s.acc & 255)
            s.acc >>= 8
            s.n -= 8

    def align(s):
        if s.n:
            s.out.append(s.acc & 255)
            s.acc = s.n = 0


def encode_row(bw, row):                # row = b"\0" + RGB bytes
    bw.put(0b010, 3)                    # BFINAL 0, BTYPE 01
    a = np.frombuffer(row, np.uint8)
    n = len(a)
    eq = np.zeros(n, bool)
    eq[4:] = a[4:] == a[1:-3]
    i = 0
    while i < n:
        if eq[i]:
            j = i
            while j < n and eq[j]:
                j += 1
            R = j - i
            while R >= 3:
                L = min(R, 258)
                bw.put(*length_code(L))
                bw.put(*DIST3)
                R -= L
                i += L
            for _ in range(R):
                bw.put(*FC[a[i]])
                i += 1
        else:
            bw.put(*FC[a[i]])
            i += 1
    bw.put(*FC[256])
    bw.put(0, 3)
    bw.align()
    bw.out += b"\x00\x00\xff\xff"


def chunk(t, d):
    return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d))


def encode(rgb, band=BAND):             # rgb: (h, w, 3) uint8
    rgb = np.ascontiguousarray(rgb, np.uint8)
    h, w, _ = rgb.shape
    out = [SIGNATURE, chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)), chunk(b"IDAT", b"\x78\x01")]
    adler = 1
    for r0 in range(0, h, band):
        bw = Bits()
        for r in range(r0, min(h, r0 + band)):
            row = b"\x00" + rgb[r].tobytes()
            encode_row(bw, row)
            adler = zlib.adler32(row, adler)
        out.append(chunk(b"IDAT", bytes(bw.out)))
    bw = Bits()
    bw.put(0b011, 3)
    bw.put(*FC[256])
    bw.align()
    out += [chunk(b"IDAT", bytes(bw.out) + struct.pack(">I", adler)), chunk(b"IEND", b"")]
    return b"".join(out)


def bound(w, h):
    """rt_png_bound's arithmetic: every raw-row byte at most 9 bits, plus the row's framing, the chunks and the
    fixed parts of the file."""
    n = 1 + 3 * w
    piece = (3 + 9 * n + 10 + 7) // 8 + 4
    bands = (h + BAND - 1) // BAND
    return 8 + 25 + 14 + 12 * bands + h * piece + 18 + 12


def chunks(png):
    """Walk a PNG's chunks, checking the signature, every length and every CRC: [(type, data), ...]."""
    assert png[:8] == SIGNATURE, "bad signature"
    i, out = 8, []
    while i < len(png):
        assert i + 12 <= len(png), "truncated chunk at byte %d" % i
        n = struct.unpack(">I", png[i:i + 4])[0]
        t = png[i + 4:i + 8]
        d = png[i + 8:i + 8 + n]
        assert len(d) == n, "truncated %r chunk" % t
        crc = struct.unpack(">I", png[i + 8 + n:i + 12 + n])[0]
        assert crc == zlib.crc32(t + d), "CRC of %r chunk at byte %d" % (t, i)
        out.append((t, d))
        i += 12 + n
        if t == b"IEND":
            break
    assert i == len(png), "bytes after IEND"
    return out


def decode(png):
    """(h, w, 3) uint8 of a colour-type-2, 8-bit, non-interlaced PNG whose rows all use filter 0 (what this
    project writes); zlib.decompress checks the Adler-32."""
    cs = chunks(png)
    assert cs[0][0] == b"IHDR" and cs[-1] == (b"IEND", b"")
    w, h, depth, ctype, comp, filt, interlace = struct.unpack(">IIBBBBB", cs[0][1])
    assert (depth, ctype, comp, filt, interlace) == (8, 2, 0, 0, 0)
    raw = zlib.decompress(b"".join(d for t, d in cs if t == b"IDAT"))
    assert len(raw) == h * (1 + 3 * w)
    rows = np.frombuffer(raw, np.uint8).reshape(h, 1 + 3 * w)
    assert not rows[:, 0].any(), "a row uses a filter other than 0"
    return rows[:, 1:].reshape(h, w, 3).copy()
