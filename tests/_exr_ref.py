"""Reference encoder and decoder of the OpenEXR layout rt_encode_exr writes.  TEST INFRASTRUCTURE.

The layout (DESIGN.md "OpenEXR output", rust-tracer_b200/csrc/rt_exr.cu): single-part scanline OpenEXR 2, ZIP
compression (16 scanlines per chunk), increasing Y, every channel FLOAT; A B G R from the float pixel {r, g, b, alpha},
and with the AOV frame also Z, coverage.Y, normal.X/Y/Z and position.X/Y/Z.  A chunk's bytes are split into even then
odd bytes and predicted (d[i] = t[i] - t[i-1] + 128); the zlib stream of d is pieces of 16 KiB, each a fixed-Huffman
block of literals and matches of distance 1 (near runs) and D2 = 2W (far runs) by a closed-form rule, then an empty
stored block; a chunk whose stream would not be smaller than its raw bytes is stored raw.  There is exactly one
byte string per image, so the GPU output is compared with `encode` byte for byte.
"""
import struct
import zlib

import numpy as np

from _png_ref import FC, LB, LE, Bits, rev

LINES = 16
PIECE = 16384
NAMES = ["A", "B", "G", "R", "Z", "coverage.Y", "normal.X", "normal.Y", "normal.Z", "position.X", "position.Y",
         "position.Z"]
# (frame, component) of each channel: 0 = the float colour pixel {r, g, b, alpha}, 1 = the AOV pixel
# {nx, ny, nz, coverage, distance, px, py, pz}
SOURCES = [(0, 3), (0, 2), (0, 1), (0, 0), (1, 4), (1, 3), (1, 0), (1, 1), (1, 2), (1, 5), (1, 6), (1, 7)]
MAGIC = 20000630

_FC_CODE = np.array([c for c, _ in FC], np.int64)
_FC_BITS = np.array([n for _, n in FC], np.int64)
_LEN_CODE = np.zeros(259, np.int64)
_LEN_BITS = np.zeros(259, np.int64)
for _L in range(3, 259):
    _k = max(k for k in range(29) if LB[k] <= _L)
    _c, _n = FC[257 + _k]
    _LEN_CODE[_L], _LEN_BITS[_L] = _c | ((_L - LB[_k]) << _n), _n + LE[_k]


def dist_code(D):
    """Distance D (1..32768) as (code with its extra bits, LSB-first, bit count): RFC 1951 3.2.5."""
    if D <= 4:
        return rev(D - 1, 5), 5
    d = D - 1
    top = d.bit_length() - 1
    e = top - 1
    code = 2 * top + ((d >> e) & 1)
    return rev(code, 5) | ((d & ((1 << e) - 1)) << 5), 5 + e


def channel_planes(rgba, aov=None):
    """The (h, w) float32 planes of the file's channels, in name order."""
    frames = [np.asarray(rgba, np.float32)] + ([] if aov is None else [np.asarray(aov, np.float32)])
    return [frames[f][..., k] for f, k in SOURCES[:4 if aov is None else 12]]


def _attr(name, typ, value):
    return name.encode() + b"\0" + typ.encode() + b"\0" + struct.pack("<i", len(value)) + value


def header(w, h, nch):
    chl = b"".join(n.encode() + b"\0" + struct.pack("<iB3xii", 2, 0, 1, 1) for n in NAMES[:nch]) + b"\0"
    box = struct.pack("<iiii", 0, 0, w - 1, h - 1)
    return (struct.pack("<II", MAGIC, 2) + _attr("channels", "chlist", chl) + _attr("compression", "compression", b"\3")
            + _attr("dataWindow", "box2i", box) + _attr("displayWindow", "box2i", box)
            + _attr("lineOrder", "lineOrder", b"\0") + _attr("pixelAspectRatio", "float", struct.pack("<f", 1.0))
            + _attr("screenWindowCenter", "v2f", struct.pack("<ff", 0.0, 0.0))
            + _attr("screenWindowWidth", "float", struct.pack("<f", 1.0)) + b"\0")


def predict(raw):
    """ZIP's split (even bytes, then odd) and predictor: d (uint8)."""
    r = np.frombuffer(raw, np.uint8)
    t = np.concatenate((r[0::2], r[1::2])).astype(np.int32)
    d = t.copy()
    d[1:] = (t[1:] - t[:-1] + 128) & 255
    return d.astype(np.uint8)


def unpredict(d):
    d = np.asarray(d, np.uint8).astype(np.int64)
    t = d.copy()
    t[1:] = d[1:] - 128
    t = np.cumsum(t) & 255
    r = np.empty(len(t), np.uint8)
    half = (len(t) + 1) // 2
    r[0::2], r[1::2] = t[:half], t[half:]
    return r.tobytes()


def _runs(mask):
    """Maximal runs of `mask` cut at piece boundaries: (starts, ends)."""
    n = len(mask)
    prev = np.zeros(n, bool)
    prev[1:] = mask[:-1]
    prev[::PIECE] = False
    nxt = np.zeros(n, bool)
    nxt[:-1] = mask[1:]
    nxt[PIECE - 1::PIECE] = False
    return np.flatnonzero(mask & ~prev), np.flatnonzero(mask & ~nxt) + 1


def _cover(starts, ends, n):
    acc = np.zeros(n + 1, np.int64)
    np.add.at(acc, starts, 1)
    np.add.at(acc, ends, -1)
    return np.cumsum(acc[:n]) > 0


def zlib_stream(d, d2, pieces=False):
    """The chunk's zlib stream by the parse rule (d2 = 0: no far distance); with `pieces`, also the offset of each
    piece in it."""
    n = len(d)
    far = np.zeros(n, bool)
    if d2:
        far[d2:] = d[d2:] == d[:-d2]
    fs, fe = _runs(far)
    keep = fe - fs >= 3
    fs, fe = fs[keep], fe[keep]
    near = np.zeros(n, bool)
    near[1:] = d[1:] == d[:-1]
    near &= ~_cover(fs, fe, n)
    ns, ne = _runs(near)
    S = np.concatenate((fs, ns))
    R = np.concatenate((fe - fs, ne - ns))
    dc, db = zip(dist_code(d2) if d2 else (0, 0), dist_code(1))
    kind = np.concatenate((np.zeros(len(fs), np.int64), np.ones(len(ns), np.int64)))
    dcode, dbits = np.array(dc, np.int64)[kind], np.array(db, np.int64)[kind]
    q, rr = R // 258, R % 258
    # matches of 258, then the tail match where R mod 258 >= 3
    run = np.repeat(np.arange(len(S)), q)
    k = np.arange(len(run)) - np.repeat(np.cumsum(q) - q, q)
    tail = np.flatnonzero(rr >= 3)
    mpos = np.concatenate((S[run] + 258 * k, S[tail] + 258 * q[tail]))
    mlen = np.concatenate((np.full(len(run), 258, np.int64), rr[tail]))
    mrun = np.concatenate((run, tail))
    mcode = _LEN_CODE[mlen] | (dcode[mrun] << _LEN_BITS[mlen])
    mbits = _LEN_BITS[mlen] + dbits[mrun]
    covered = _cover(S, S + 258 * q + np.where(rr >= 3, rr, 0), n)
    lpos = np.flatnonzero(~covered)
    pos = np.concatenate((mpos, lpos))
    code = np.concatenate((mcode, _FC_CODE[d[lpos]]))
    bits = np.concatenate((mbits, _FC_BITS[d[lpos]]))
    order = np.argsort(pos, kind="stable")
    pos, code, bits = pos[order], code[order], bits[order]
    piece = pos // PIECE
    npieces = (n + PIECE - 1) // PIECE
    piece_bits = 3 + np.bincount(piece, weights=bits, minlength=npieces).astype(np.int64)
    piece_len = (piece_bits + 17) // 8 + 4
    piece_off = 2 + np.concatenate(([0], np.cumsum(piece_len)[:-1]))
    excl = np.cumsum(bits) - bits
    first = np.searchsorted(piece, np.arange(npieces))
    local = excl - excl[np.minimum(first, len(excl) - 1)][piece] if len(excl) else excl
    bitpos = 8 * piece_off[piece] + 3 + local
    total = 2 + int(piece_len.sum()) + 6
    out = np.zeros(total, np.float64)
    v = code << (bitpos & 7)
    for b in range(5):
        out += np.bincount((bitpos >> 3) + b, weights=((v >> (8 * b)) & 255).astype(np.float64), minlength=total)[:total]
    out = out.astype(np.uint8)
    out[piece_off] |= 2                      # BFINAL 0, BTYPE 01
    out[piece_off + piece_len - 2] = 0xFF    # the empty stored block's NLEN
    out[piece_off + piece_len - 1] = 0xFF
    out[0], out[1] = 0x78, 0x01
    out[-6:] = np.frombuffer(b"\x03\x00" + struct.pack(">I", zlib.adler32(d.tobytes())), np.uint8)
    return (out.tobytes(), piece_off) if pieces else out.tobytes()


def slow_stream(d, d2):
    """The zlib stream of one chunk by the parse rule, byte by byte (for small inputs)."""
    d = [int(v) for v in d]
    n = len(d)
    out = bytearray(b"\x78\x01")
    for p0 in range(0, n, PIECE):
        p1 = min(n, p0 + PIECE)
        far = [bool(d2) and i >= d2 and d[i] == d[i - d2] for i in range(p0, p1)]
        in_far = [False] * (p1 - p0)
        i = 0
        while i < len(far):
            j = i
            while j < len(far) and far[j]:
                j += 1
            if j - i >= 3:
                in_far[i:j] = [True] * (j - i)
            i = max(j, i + 1)
        near = [(p0 + k) >= 1 and d[p0 + k] == d[p0 + k - 1] and not in_far[k] for k in range(p1 - p0)]
        bw = Bits()
        bw.put(0b010, 3)
        k = 0
        while k < p1 - p0:
            mask = in_far if in_far[k] else near if near[k] else None
            if mask is None:
                bw.put(*FC[d[p0 + k]])
                k += 1
                continue
            dc = dist_code(d2 if mask is in_far else 1)
            j = k
            while j < p1 - p0 and mask[j]:
                j += 1
            R = j - k
            for _ in range(R // 258):
                bw.put(int(_LEN_CODE[258]), int(_LEN_BITS[258]))
                bw.put(*dc)
            rr = R % 258
            if rr >= 3:
                bw.put(int(_LEN_CODE[rr]), int(_LEN_BITS[rr]))
                bw.put(*dc)
            else:
                for q in range(j - rr, j):
                    bw.put(*FC[d[p0 + q]])
            k = j
        bw.put(*FC[256])
        bw.put(0, 3)
        bw.align()
        out += bw.out + b"\x00\x00\xff\xff"
    return bytes(out) + b"\x03\x00" + struct.pack(">I", zlib.adler32(bytes(d)))


def chunk_raw(planes, y0, y1):
    return b"".join(p[y].astype("<f4").tobytes() for y in range(y0, y1) for p in planes)


def encode(rgba, aov=None):
    """The file of a float frame (h, w, 4) and, optionally, its AOV frame (h, w, 8)."""
    planes = channel_planes(rgba, aov)
    h, w = planes[0].shape
    d2 = 2 * w if 2 * w <= 32768 else 0
    head = header(w, h, len(planes))
    chunks = []
    for y0 in range(0, h, LINES):
        raw = chunk_raw(planes, y0, min(h, y0 + LINES))
        z = zlib_stream(predict(raw), d2)
        data = z if len(z) < len(raw) else raw
        chunks.append(struct.pack("<ii", y0, len(data)) + data)
    off = len(head) + 8 * len(chunks)
    table = b""
    for c in chunks:
        table += struct.pack("<Q", off)
        off += len(c)
    return head + table + b"".join(chunks)


def bound(w, h, aov=False):
    """rt_exr_bound's arithmetic: the header, the offset table and every chunk stored raw."""
    nch = 12 if aov else 4
    chunks = (h + LINES - 1) // LINES
    return len(header(w, h, nch)) + 16 * chunks + h * w * nch * 4


def decode(data):
    """{channel name: (h, w) float32} of a file of this layout, checking the header and every chunk; a chunk is raw
    when its size is its uncompressed size, else one zlib stream (zlib.decompress checks the Adler-32)."""
    assert struct.unpack("<II", data[:8]) == (MAGIC, 2)
    i, attrs = 8, {}
    while data[i] != 0:
        name, i = data[i:data.index(b"\0", i)].decode(), data.index(b"\0", i) + 1
        typ, i = data[i:data.index(b"\0", i)].decode(), data.index(b"\0", i) + 1
        size = struct.unpack("<i", data[i:i + 4])[0]
        attrs[name] = (typ, data[i + 4:i + 4 + size])
        i += 4 + size
    i += 1
    assert list(attrs) == ["channels", "compression", "dataWindow", "displayWindow", "lineOrder", "pixelAspectRatio",
                           "screenWindowCenter", "screenWindowWidth"]
    assert attrs["compression"] == ("compression", b"\3") and attrs["lineOrder"] == ("lineOrder", b"\0")
    x0, y0_, x1, y1 = struct.unpack("<iiii", attrs["dataWindow"][1])
    assert (x0, y0_) == (0, 0) and attrs["displayWindow"] == attrs["dataWindow"]
    w, h = x1 + 1, y1 + 1
    chl, names, j = attrs["channels"][1], [], 0
    while chl[j] != 0:
        e = chl.index(b"\0", j)
        names.append(chl[j:e].decode())
        assert struct.unpack("<iB3xii", chl[e + 1:e + 17]) == (2, 0, 1, 1)
        j = e + 17
    assert names == sorted(names, key=str.encode)
    nch, chunks = len(names), (h + LINES - 1) // LINES
    table = struct.unpack("<%dQ" % chunks, data[i:i + 8 * chunks])
    out = np.empty((nch, h, w), np.float32)
    end = i + 8 * chunks
    for c, off in enumerate(table):
        assert off == end, "chunk %d at %d, expected %d" % (c, off, end)
        y0, size = struct.unpack("<ii", data[off:off + 8])
        rows = min(LINES, h - y0)
        assert y0 == c * LINES
        n = rows * nch * w * 4
        body = data[off + 8:off + 8 + size]
        raw = body if size == n else unpredict(np.frombuffer(zlib.decompress(body), np.uint8))
        assert len(raw) == n
        out[:, y0:y0 + rows] = np.frombuffer(raw, "<f4").reshape(rows, nch, w).transpose(1, 0, 2)
        end = off + 8 + size
    assert end == len(data), "bytes after the last chunk"
    return {name: out[k] for k, name in enumerate(names)}


def chunk_kinds(data):
    """Per chunk: True when stored raw, False when compressed."""
    planes = decode(data)
    nch = len(planes)
    h, w = next(iter(planes.values())).shape
    i = data.index(b"screenWindowWidth") + len("screenWindowWidth") + 1 + 6 + 4 + 4 + 1
    chunks = (h + LINES - 1) // LINES
    table = struct.unpack("<%dQ" % chunks, data[i:i + 8 * chunks])
    kinds = []
    for off in table:
        y0, size = struct.unpack("<ii", data[off:off + 8])
        kinds.append(size == min(LINES, h - y0) * nch * w * 4)
    return kinds
