"""rt_encode_exr on frames built from chosen predicted bytes: the parse rule's edges, every far distance, files that
mix raw and compressed chunks (and the tie between them), scratch reuse, and a file whose offsets pass 2^32.

Rendered frames always compress and noise never does, so those alone leave most of the encoder's paths unrun.  Here
each case is a list of predicted streams d, one per chunk, written segment by segment (literals, near runs, far runs
at chosen positions); `frames_from_predicted` inverts ZIP's predictor and split to get the float frames whose chunks
predict back to exactly those streams.  Such frames are full of NaNs with arbitrary payloads and subnormals (and
`special_floats` adds +-0 and +-inf), so they also check that every float is carried bit for bit: frames go to the
device as int32 and are compared as uint32.

The CPU part checks every case's stream against the byte-by-byte statement of the parse rule, zlib and the
reference decoder, and that the case set still reaches every edge it is meant to (`test_cases_cover_the_edges`); the
GPU part compares the device's file with the reference's byte for byte, and on a mismatch names the chunk, the piece
and the first differing byte.

Run as a script (`python test_exr_edges.py past-4-gib`) it encodes the 4.3 GB frame of `test_file_past_4_gib` in a
process of its own, so that the encoder's scratch for it goes back to the device when that process ends."""
import os

os.environ["OPENCV_IO_ENABLE_OPENEXR"] = "1"   # before OpenCV is imported anywhere

import functools
import json
import random
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == "__main__":
    sys.path[:0] = [HERE, os.path.join(os.path.dirname(HERE), "rust-tracer_b200")]

import _exr_ref as X

PIECE, LINES = X.PIECE, X.LINES
SLOW_MAX = 65536   # streams up to this length are also checked against X.slow_stream


def nch_of(aov):
    return 12 if aov else 4


def d2_of(w):
    return 2 * w if 2 * w <= 32768 else 0


def chunk_sizes(w, h, aov):
    """Predicted bytes of each chunk."""
    return [min(LINES, h - y0) * nch_of(aov) * 4 * w for y0 in range(0, h, LINES)]


def dist_code(D):
    """Deflate distance code (0..29) of distance D."""
    if D <= 4:
        return D - 1
    d = D - 1
    top = d.bit_length() - 1
    return 2 * top + ((d >> (top - 1)) & 1)


# ---- frames from predicted streams --------------------------------------------------------------------------------
def frames_from_predicted(streams, w, h, aov):
    """The (h, w, 4) colour frame and, for 12 channels, the (h, w, 8) AOV frame (else None), as uint32 bit patterns,
    whose chunk c predicts to streams[c]."""
    nch = nch_of(aov)
    planes = np.empty((nch, h, w), np.uint32)
    for c, d in enumerate(streams):
        y0 = c * LINES
        rows = min(LINES, h - y0)
        raw = np.frombuffer(X.unpredict(d), "<u4")
        assert raw.size == rows * nch * w, (c, raw.size)
        planes[:, y0:y0 + rows] = raw.reshape(rows, nch, w).transpose(1, 0, 2)
    frames = [np.zeros((h, w, 4), np.uint32), np.zeros((h, w, 8), np.uint32) if aov else None]
    for k, (f, comp) in enumerate(X.SOURCES[:nch]):
        frames[f][..., comp] = planes[k]
    return frames[0], frames[1]


def as_float(frame):
    return None if frame is None else frame.view(np.float32)


class Stream:
    """A predicted stream of n bytes with far distance d2, written left to right.  Literals never equal the byte
    before them or the byte d2 before them, so they end any run and start none."""

    def __init__(self, n, d2, seed):
        self.d, self.n, self.d2, self.i = bytearray(n), n, d2, 0
        self.rng = random.Random(seed)

    def _banned(self, i):
        b = {self.d[i - 1]} if i else set()
        if self.d2 and i >= self.d2:
            b.add(self.d[i - self.d2])
        return b

    def lit(self, k, lo=0, hi=256):
        """k literals in [lo, hi)."""
        for _ in range(k):
            banned = self._banned(self.i)
            v = self.rng.randrange(lo, hi)
            while v in banned:
                v = self.rng.randrange(lo, hi)
            self.d[self.i] = v
            self.i += 1
        return self

    def near(self, R, lo=0, hi=256):
        """A literal, then a near run of R bytes equal to it (none of them equal to its byte d2 back)."""
        i = self.i
        banned = self._banned(i)
        if self.d2:
            banned |= {self.d[j - self.d2] for j in range(max(i, self.d2), min(i + R + 1, i + self.d2))}
        v = self.rng.randrange(lo, hi)
        while v in banned:
            v = self.rng.randrange(lo, hi)
        self.d[i:i + R + 1] = bytes([v]) * (R + 1)
        self.i += R + 1
        return self

    def rep(self, R):
        """R more bytes equal to the last one."""
        self.d[self.i:self.i + R] = bytes([self.d[self.i - 1]]) * R
        self.i += R
        return self

    def far(self, R):
        """R bytes copying the byte d2 back."""
        assert self.d2 and self.i >= self.d2
        while R:
            k = min(R, self.d2)
            self.d[self.i:self.i + k] = self.d[self.i - self.d2:self.i - self.d2 + k]
            self.i += k
            R -= k
        return self

    def put(self, values):
        self.d[self.i:self.i + len(values)] = bytes(values)
        self.i += len(values)
        return self

    def to(self, p, lo=0, hi=256):
        """Literals up to position p."""
        assert p >= self.i, (p, self.i)
        return self.lit(p - self.i, lo, hi)

    def lane(self, r, lo=0, hi=256):
        """Literals up to the next position that is r mod 32."""
        return self.lit((r - self.i) % 32, lo, hi)

    def fill(self, lo=0, hi=256):
        return self.to(self.n, lo, hi)

    def done(self):
        assert self.i == self.n, (self.i, self.n)
        return np.frombuffer(bytes(self.d), np.uint8)


# ---- the cases --------------------------------------------------------------------------------------------------
RUN_LENGTHS = [1, 2, 3, 4, 257, 258, 259, 260, 261, 515, 516, 517, 518, 519, 774]
RUN_LANES = [0, 1, 29, 30, 31]
MIXED = [3, 4, 5, 9, 30, 100, 227, 257, 258, 259, 260, 261, 300, 516, 517, 518, 700, 1000]
CASES = {}   # name -> (w, h, aov, builder of the streams, expected kinds or None)


def case(name, w, h, aov, kinds=None):
    def reg(fn):
        CASES[name] = (w, h, aov, fn, kinds)
        return fn
    return reg


def streams_for(w, h, aov, seed, body):
    """One Stream per chunk, each handed to body(stream, chunk index) and completed with literals."""
    out = []
    for c, n in enumerate(chunk_sizes(w, h, aov)):
        s = Stream(n, d2_of(w), seed * 1000 + c)
        body(s, c)
        out.append(s.fill().done())
    return out


@case("run_lengths", 256, 32, False)
def _run_lengths():
    """Near (chunk 0) and far (chunk 1) runs of every length in RUN_LENGTHS, starting at lanes 0, 1, 29, 30, 31."""
    def body(s, c):
        s.lit(s.d2 + 40)
        for R in RUN_LENGTHS:
            for r in RUN_LANES:
                if c == 0:
                    s.lane((r - 1) % 32).near(R).lit(2)
                else:
                    s.lane(r).far(R).lit(2)
    return streams_for(256, 32, False, 1, body)


@case("far_priority", 64, 16, False)
def _far_priority():
    """D2 = 128.  Background literals are < 100, special bytes >= 100."""
    def body(s, c):
        s.lit(s.d2, 0, 100).far(5).lit(3, 0, 100)              # a far run at i = D2, the first eligible byte
        p = s.i                                                  # a far pair inside a near run: near wins
        s.lit(2, 0, 100).put([200, 200]).lit(4, 0, 100).to(p + s.d2, 0, 100)
        s.lit(1, 0, 100).put([200] * 6).lit(4, 0, 100)
        p = s.i                                                  # a far run of 3 inside a near run: far wins,
        s.lit(2, 0, 100).put([201] * 3).lit(3, 0, 100).to(p + s.d2, 0, 100)   # then a near run of 2
        s.lit(1, 0, 100).put([201] * 6).lit(4, 0, 100)
        for r in (29, 30, 31):                                   # far runs of 3 at mask bits 29, 30, 31
            s.lane(r, 0, 100).far(3).lit(3, 0, 100)
            s.lane(r, 0, 100).far(4).lit(3, 0, 100)
        s.near(7, 100, 256).far(9).lit(2, 0, 100)                # a near run directly followed by a far run
        s.far(9).rep(7).lit(2, 0, 100)                           # and the reverse
        s.far(300).near(300, 100, 256).far(3).rep(3).lit(1, 0, 100)
        s.lit(1, 100, 143)
        for v in (0, 143, 144, 255, 1, 142, 145, 254):           # literal values at the 8/9-bit edges
            s.put([v]).lit(1, 100, 143)
        s.far(258 * 3 + 1).lit(1).far(258 * 2 + 2).lit(1).far(258 + 3).lit(1)
    return streams_for(64, 16, False, 2, body)


BOUNDARY = [(a, b) for a in range(4) for b in range(4) if a + b] + [(300, 300)]


@case("piece_boundaries", 64, 256, True)
def _piece_boundaries():
    """12 channels, 3 pieces per chunk: near and far runs with a bytes before and b after each piece boundary."""
    configs = [("near", a, b) for a, b in BOUNDARY] + [("far", a, b) for a, b in BOUNDARY]

    def body(s, c):
        s.lit(s.d2).far(20).lit(2).near(20).lit(2)
        for j in (1, 2):
            kind, a, b = configs[2 * c + j - 1]
            P = j * PIECE
            if kind == "near":
                s.to(P - a - 1).near(a + b)
            else:
                s.to(P - a).far(a + b)
            s.lit(2).near(5).lit(1).far(6).lit(1)
    return streams_for(64, 256, True, 3, body)


@case("whole_piece_runs", 8192, 1, False)
def _whole_piece_runs():
    """D2 = 16384, so piece 1 starts at i = D2: piece 1 is one near run, piece 3 one far run (63 x 258 + 130)."""
    def body(s, c):
        s.lit(PIECE - 1, 0, 100).near(PIECE, 100, 256)
        s.to(3 * PIECE, 0, 100).far(PIECE)
        s.to(4 * PIECE).put([9] * PIECE)
        while s.i < s.n - 1200:
            s.far(s.rng.choice(MIXED)).lit(s.rng.randrange(1, 4))
    return streams_for(8192, 1, False, 4, body)


@case("constant_chunks", 64, 32, True)
def _constant_chunks():
    """A chunk whose predicted bytes are all equal, and one whose raw bytes are."""
    n = chunk_sizes(64, 32, True)[0]
    return [np.full(n, 7, np.uint8), X.predict(b"\x3f" * n)]


def split_body(s, c):
    """Runs around the split point n/2, far runs whose partner is across it, runs in the short last piece."""
    h = s.n // 2
    s.lit(s.d2).far(40).lit(1)
    if (s.n // 16) % 2:                                 # odd W: a near run across n/2, even W: a far run
        s.to(h - 20).near(40).lit(1)
    else:
        s.to(h - 17).far(40).lit(1)
    s.to(h + 200).far(40).lit(1)
    s.to(h + s.d2 - 30).far(60).lit(1)                  # partners of h + d2 - 30 .. h + d2 - 1 are below n/2
    s.to(h + 2 * s.d2 - 5).far(10).lit(1)
    last = s.n - (s.n % PIECE or PIECE)
    s.to(last - 3).far(7).lit(1).near(4).lit(1).far(3)
    if s.n - s.i > 20:
        s.lit(1).near(min(12, s.n - s.i - 2))


for _w in (1025, 1026, 1027):
    case("split_mid_step_w%d" % _w, _w, 1, False)(lambda _w=_w: streams_for(_w, 1, False, _w, split_body))


@case("split_on_piece_boundary", 128, 32, False)
def _split_on_piece_boundary():
    """n/2 = 16384 is the first piece boundary: a near run (chunk 0) and a far run (chunk 1) across it."""
    def body(s, c):
        h = s.n // 2
        s.lit(s.d2).far(30).lit(1)
        if c == 0:
            s.to(h - 9).near(20)
        else:
            s.to(h - 11).far(25)
        s.lit(1).far(300).lit(1).near(260)
    return streams_for(128, 32, False, 6, body)


@case("nine_bit_piece", 128, 16, False)
def _nine_bit_piece():
    """Piece 0 is 16,384 9-bit literals (3 + 9 * 16384 bits, the largest slot), piece 1 one run, so the chunk still
    compresses and the worst-case slot is copied into the file."""
    return streams_for(128, 16, False, 7, lambda s, c: s.lit(PIECE, 144, 256).near(PIECE - 1, 0, 144))


@case("long_tokens", 16384, 2, False)
def _long_tokens():
    """D2 = 32768 (13 extra bits): far runs with R mod 258 in [227, 257], whose tail token is 31 bits, between 1..40
    mixed literals, so those tokens land at every bit offset of the window."""
    def body(s, c):
        s.lit(s.d2)
        while s.i < s.n - 1000:
            s.far(258 * s.rng.randrange(3) + s.rng.randrange(227, 258)).lit(s.rng.randrange(1, 41))
    return streams_for(16384, 2, False, 8, body)


FAR_WIDTHS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 12, 13, 16, 17, 24, 25, 32, 33, 48, 49, 64, 65, 96, 97, 128, 129, 192, 193,
              256, 257, 384, 385, 512, 513, 768, 769, 1024, 1025, 1536, 1537, 2048, 2049, 3072, 3073, 4096, 4097,
              6144, 6145, 8192, 8193, 12288, 12289, 16384, 16385]


def far_body(s, c):
    if not s.d2:   # W = 16385: no far distance, so near runs
        while s.n - s.i > 5:
            s.near(min(s.rng.choice(MIXED), s.n - s.i - 5)).lit(s.rng.randrange(1, 4))
        return
    s.lit(min(s.d2, s.n))
    while s.n - s.i > 4:
        s.far(min(s.rng.choice(MIXED), s.n - s.i - 4)).lit(s.rng.randrange(1, 4))


for _w in FAR_WIDTHS:
    for _aov in (False, True):
        case("far_w%d_%dch" % (_w, nch_of(_aov)), _w, 3, _aov)(
            lambda _w=_w, _aov=_aov: streams_for(_w, 3, _aov, 9, far_body))


def raw_body(s, c):
    pass   # only literals of the full range: 8.44 bits a byte, so the stream is longer than the raw bytes


def packed_body(s, c):
    if s.n < s.d2:   # W = 64: every chunk is longer than D2
        return
    s.lit(s.d2)
    while s.n - s.i > 12:
        s.far(min(s.rng.choice(MIXED), s.n - s.i - 12)).lit(s.rng.randrange(1, 6))
        s.near(min(s.rng.choice(MIXED[:8]), s.n - s.i - 2)).lit(1)


for _pat in ("CRCR", "RCRC", "RRRC", "CCCR"):
    for _aov in (False, True):
        def _mixed(pat=_pat, aov=_aov):
            bodies = [packed_body if k == "C" else raw_body for k in pat]
            return streams_for(64, 53, aov, 10, lambda s, c: bodies[c](s, c))
        case("kinds_%s_%dch" % (_pat, nch_of(_aov)), 64, 53, _aov, [k == "R" for k in _pat])(_mixed)


SPECIAL = [0x00000000, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00001, 0x7F800001, 0x7FBFFFFF,
           0x00000001, 0x807FFFFF, 0x00400000, 0x7F7FFFFF]   # +-0, +-inf, NaNs, subnormals, the largest float


@case("special_floats", 33, 20, True)
def _special_floats():
    """Streams of frames made of +-0, +-inf, quiet and signalling NaNs with payloads, subnormals and the largest
    float, some in runs along x."""
    planes = np.array(SPECIAL, np.uint32)[np.random.default_rng(13).integers(0, len(SPECIAL), (12, 20, 33))]
    planes[:, :, 10:20] = planes[:, :, 10:11]
    return [X.predict(planes[:, y0:y0 + LINES].transpose(1, 0, 2).astype("<u4").tobytes()) for y0 in (0, LINES)]


@functools.lru_cache(None)
def tie_streams():
    """Streams of n - 1, n and n + 1 zlib bytes for a chunk of n = 16384 (W = 64, 4 channels): a leading run of L
    bytes, then full-range literals; L is searched, deterministically."""
    n, d2 = 16384, 128
    tail = Stream(n, d2, 12).lit(n).done()

    def stream(L):
        d = np.concatenate((np.full(L + 1, tail[0] ^ 0x55, np.uint8), tail[:n - L - 1]))
        return d, len(X.zlib_stream(d, d2))

    lo, hi = 0, n // 2                    # the stream shrinks as L grows: find where it crosses n
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if stream(mid)[1] > n else (lo, mid)
    found = {}
    for L in range(max(0, lo - 100), lo + 100):
        d, z = stream(L)
        if z - n in (-1, 0, 1):
            found.setdefault(z - n, d)
    assert sorted(found) == [-1, 0, 1], sorted(found)
    return found[-1], found[0], found[1]


@case("tie_first_chunk", 64, 16, False, [True])
def _tie_first():
    return [tie_streams()[1]]


@case("tie_three_chunks", 64, 48, False, [False, True, True])
def _tie_three():
    return list(tie_streams())


@case("tie_in_mixed_file", 64, 53, False, [False, True, True, False])
def _tie_mixed():
    s = streams_for(64, 53, False, 12, lambda s, c: (packed_body if c in (0, 3) else raw_body)(s, c))
    return [s[0], tie_streams()[1], s[2], s[3]]


class Case:
    """Streams, one per chunk, of a w x h frame (12 channels with aov), the frames they come from and the reference's
    file; `kinds`: the raw (True) or compressed kind expected of each chunk, when the case is about it."""

    def __init__(self, name, w, h, aov, streams, kinds=None):
        self.name, self.w, self.h, self.aov, self.streams, self.kinds = name, w, h, aov, streams, kinds
        self.d2 = d2_of(w)
        self.rgba, self.aovf = frames_from_predicted(streams, w, h, aov)

    @functools.cached_property
    def file(self):
        return X.encode(as_float(self.rgba), as_float(self.aovf))


@functools.lru_cache(None)
def get(name):
    w, h, aov, fn, kinds = CASES[name]
    return Case(name, w, h, aov, fn(), kinds)


def parse(d, d2):
    """The reference's parse of one stream: far runs and near runs as (starts, ends), cut at piece boundaries."""
    n = len(d)
    far = np.zeros(n, bool)
    if d2:
        far[d2:] = d[d2:] == d[:-d2]
    fs, fe = X._runs(far)
    keep = fe - fs >= 3
    fs, fe = fs[keep], fe[keep]
    near = np.zeros(n, bool)
    near[1:] = d[1:] == d[:-1]
    near &= ~X._cover(fs, fe, n)
    ns, ne = X._runs(near)
    return (fs, fe), (ns, ne), far, near


# ---- comparing files ----------------------------------------------------------------------------------------------
def table_of(data, w, h, aov):
    chunks = (h + LINES - 1) // LINES
    at = len(X.header(w, h, nch_of(aov)))
    return np.frombuffer(data[at:at + 8 * chunks], "<u8").astype(np.int64)


def assert_same_file(got, c):
    """got == c.file, else a message naming the chunk, its kind, the piece and the first differing byte."""
    want = c.file
    if got == want:
        return
    m = min(len(got), len(want))
    diff = np.flatnonzero(np.frombuffer(got[:m], np.uint8) != np.frombuffer(want[:m], np.uint8))
    k = int(diff[0]) if len(diff) else m
    table = table_of(want, c.w, c.h, c.aov)
    where = "the header or offset table"
    if k >= table[0]:
        ch = int(np.searchsorted(table, k, "right") - 1)
        q = k - int(table[ch]) - 8
        n = chunk_sizes(c.w, c.h, c.aov)[ch]
        size = struct.unpack("<i", want[table[ch] + 4:table[ch] + 8])[0]
        if q < 0:
            where = "chunk %d's y0/size" % ch
        elif size == n:
            where = "chunk %d (raw), byte %d" % (ch, q)
        else:
            _, off = X.zlib_stream(c.streams[ch], c.d2, pieces=True)
            j = int(np.searchsorted(off, q, "right") - 1)
            where = "chunk %d (compressed, %d bytes), piece %d, byte %d of the piece" % (ch, size, j, q - off[max(j, 0)])
    pytest.fail("%s: files differ first at byte %d, in %s: got %s, want %s (lengths %d, %d)" % (
        c.name, k, where, got[k:k + 1].hex() or "end", want[k:k + 1].hex() or "end", len(got), len(want)))


def cv2_reads(data, rgba, tmp_path):
    """OpenEXR through OpenCV reads the RGBA layer bit for bit (when OpenCV has EXR support)."""
    try:
        import cv2
    except ImportError:
        return
    p = str(tmp_path / "case.exr")
    with open(p, "wb") as f:
        f.write(data)
    try:
        img = cv2.imread(p, cv2.IMREAD_UNCHANGED)
    except cv2.error:
        return
    if img is None:
        return
    h, w = rgba.shape[:2]
    assert np.array_equal(img.reshape(h, w, 4).view(np.uint32), rgba[..., [2, 1, 0, 3]])


# ---- CPU ----------------------------------------------------------------------------------------------------------
NAMES = sorted(CASES)


@pytest.mark.parametrize("name", NAMES)
def test_case_reference(name, tmp_path):
    """The built frames predict back to the streams; the stream is the byte-by-byte statement's and inflates back;
    the reference's file decodes to the frames bit for bit."""
    c = get(name)
    planes = X.channel_planes(as_float(c.rgba), as_float(c.aovf))
    kinds = []
    for k, d in enumerate(c.streams):
        y0 = k * LINES
        assert np.array_equal(X.predict(X.chunk_raw(planes, y0, min(c.h, y0 + LINES))), d), "chunk %d" % k
        z = X.zlib_stream(d, c.d2)
        if len(d) <= SLOW_MAX:
            assert z == X.slow_stream(d, c.d2), "chunk %d" % k
        assert zlib.decompress(z) == d.tobytes()
        kinds.append(len(z) >= len(d))
    assert X.chunk_kinds(c.file) == kinds
    if c.kinds is not None:
        assert kinds == c.kinds
    dec = X.decode(c.file)
    assert list(dec) == X.NAMES[:nch_of(c.aov)]
    for nm, plane in zip(X.NAMES, planes):
        assert np.array_equal(dec[nm].view(np.uint32), plane.view(np.uint32)), nm
    if c.w * c.h <= 1 << 16:
        cv2_reads(c.file, c.rgba, tmp_path)


def test_frames_hold_every_kind_of_float():
    """Frames built from streams carry NaNs with payloads and subnormals, and special_floats every special value, all
    of which a float copy could change."""
    bits = np.concatenate([get(n).rgba.ravel() for n in ("run_lengths", "far_priority", "long_tokens")])
    exp, man = (bits >> 23) & 255, bits & 0x7FFFFF
    assert ((exp == 255) & (man != 0) & (man != 0x400000)).any()    # NaN, not the canonical one
    assert ((exp == 0) & (man != 0)).any()                          # subnormal
    c = get("special_floats")
    assert set(SPECIAL) <= set(np.concatenate((c.rgba.ravel(), c.aovf.ravel())).tolist())


def test_tie_is_the_raw_side():
    """Streams of n - 1, n and n + 1 bytes: compressed, raw, raw (the rule is "not smaller => raw")."""
    n = 16384
    for d, k in zip(tie_streams(), (-1, 0, 1)):
        assert len(d) == n and len(X.zlib_stream(d, 128)) == n + k
        assert len(X.slow_stream(d, 128)) == n + k


def test_cases_cover_the_edges():
    """What the cases are for, counted from the reference's own parse, so an edit to a builder cannot silently drop
    an edge."""
    lanes = {"far": set(), "near": set()}
    classes = {"far": set(), "near": set()}
    cut = {"far": 0, "near": 0}
    across_word, codes, mixed, tie, nine_bit_slot = 0, set(), 0, 0, 0
    lits = set()
    for name in NAMES:
        c = get(name)
        kinds = []
        for d in c.streams:
            n = len(d)
            (fs, fe), (ns, ne), far, near = parse(d, c.d2)
            for kind, s, e, mask in (("far", fs, fe, far), ("near", ns, ne, near)):
                lanes[kind] |= set((s % 32).tolist())
                R = e - s
                classes[kind] |= {(int(q), min(int(r), 3)) for q, r in zip(R // 258, R % 258) if q <= 2}
                # cut by a piece boundary: the mask goes on in the next piece
                cut[kind] += int(sum(1 for x in e if x % PIECE == 0 and x < n and mask[x]))
            across_word += int(((fe - fs == 3) & (fs % 32 >= 30)).sum())
            if len(fs):
                codes.add(dist_code(c.d2))
            if len(ns):
                codes.add(0)
            z = len(X.zlib_stream(d, c.d2))
            kinds.append(z >= n)
            tie += z == n
            covered = X._cover(np.concatenate((fs, ns)), np.concatenate((fe, ne)), n)
            lits |= set(np.unique(d[~covered]).tolist())
            if z < n:
                for p0 in range(0, n, PIECE):
                    if not covered[p0:p0 + PIECE].any() and (d[p0:p0 + PIECE] >= 144).all() and n - p0 >= PIECE:
                        nine_bit_slot += 1
        mixed += len(set(kinds)) == 2
    assert lanes["far"] == set(range(32)) and lanes["near"] == set(range(32))
    assert classes["near"] == {(q, r) for q in range(3) for r in range(4)} - {(0, 0)}
    assert classes["far"] == {(q, r) for q in range(3) for r in range(4)} - {(0, 0), (0, 1), (0, 2)}
    assert cut["far"] >= 8 and cut["near"] >= 8
    assert across_word >= 2
    assert codes == {0, 1} | set(range(3, 30)), sorted(set(range(30)) - codes)   # distance 1 and every even one
    assert mixed >= 8 and tie >= 3 and nine_bit_slot >= 1
    assert {0, 143, 144, 255} <= lits


def test_far_widths_sit_at_the_ends_of_every_distance_code():
    """FAR_WIDTHS holds, for every code an even distance can have, the widths whose D2 = 2W is its lowest and its
    highest even distance (and the reference's code agrees with dist_code)."""
    ends = {}
    for D in range(2, 32769, 2):
        ends.setdefault(dist_code(D), []).append(D)
    want = {D // 2 for ds in ends.values() for D in (ds[0], ds[-1])}
    assert want == {w for w in FAR_WIDTHS if d2_of(w)} and sorted(ends) == [1] + list(range(3, 30))
    for D in range(1, 32769):
        code, nbits = X.dist_code(D)
        assert code & 31 == int("{:05b}".format(dist_code(D))[::-1], 2)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def to_device(frame, pitch_floats=None):
    """A frame on the device as int32 (no float conversion touches a NaN's payload), optionally inside rows of
    pitch_floats words padded with 0xFF bytes; returns (tensor, pitch in bytes)."""
    import torch
    h, w, k = frame.shape
    src = torch.from_numpy(frame.view(np.int32).reshape(h, w * k))
    if pitch_floats is None:
        return src.cuda(), 0
    t = torch.full((h, pitch_floats), -1, dtype=torch.int32)
    t[:, :w * k] = src
    return t.cuda(), pitch_floats * 4


def encode_case(rt, c, pitch=None, aov_pitch=None):
    rgba, rp = to_device(c.rgba, pitch)
    if c.aovf is None:
        return rt.encode_exr(rgba.data_ptr(), c.w, c.h, pitch=rp)
    aov, ap = to_device(c.aovf, aov_pitch)
    return rt.encode_exr(rgba.data_ptr(), c.w, c.h, aov_ptr=aov.data_ptr(), pitch=rp, aov_pitch=ap)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_device_file_is_the_reference(rt, name):
    c = get(name)
    assert_same_file(encode_case(rt, c), c)


@pytest.mark.gpu
def test_pitched_frames_with_0xff_padding(rt):
    """A mixed file from frames in padded rows, the colour and AOV pitches differing."""
    c = get("kinds_CRCR_12ch")
    assert_same_file(encode_case(rt, c, pitch=c.w * 4 + 12, aov_pitch=c.w * 8 + 4), c)


@pytest.mark.gpu
def test_scratch_reuse_on_one_stream(rt):
    """Scratch and the output buffer are kept per (device, stream) and never cleared: a small file after a large one
    on the same stream, then the large one again, each equal to the reference."""
    rng = np.random.default_rng(21)
    big = Case("noise", 1000, 70, True, [rng.integers(0, 256, n).astype(np.uint8) for n in chunk_sizes(1000, 70, True)])
    small = get("constant_chunks")
    for c in (big, small, big, get("tie_in_mixed_file"), small):
        assert_same_file(encode_case(rt, c), c)


@pytest.mark.gpu
def test_same_frame_on_two_streams_and_device_output(rt):
    """The C ABI on two streams, with host and device output, gives the reference's file each time."""
    import torch
    c = get("kinds_RCRC_12ch")
    rgba, _ = to_device(c.rgba)
    aov, _ = to_device(c.aovf)
    L, n = rt.lib(), rt.C.c_size_t()
    cap = rt.exr_bound(c.w, c.h, True)
    host = rt.C.create_string_buffer(cap)
    dev = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()
    for s in streams:
        assert L.rt_encode_exr(rgba.data_ptr(), 0, aov.data_ptr(), 0, c.w, c.h, host, cap, rt.C.byref(n),
                               s.cuda_stream) == rt.RT_OK
        assert_same_file(host.raw[:n.value], c)
        dev.fill_(0xAB)
        torch.cuda.synchronize()
        assert L.rt_encode_exr(rgba.data_ptr(), 0, aov.data_ptr(), 0, c.w, c.h, dev.data_ptr(), cap, rt.C.byref(n),
                               s.cuda_stream) == rt.RT_OK
        s.synchronize()
        assert_same_file(bytes(dev[:n.value].cpu().numpy()), c)
        assert bool((dev[n.value:] == 0xAB).all())   # nothing written past the file


@pytest.mark.gpu
def test_file_past_4_gib(rt):
    """A 4-channel 16384 x 16400 frame (4,299,161,600 raw bytes): chunks 0-1023 are noise (raw), chunk 1024 is
    constant (compressed), so its table entry, header, data and Adler-32 sit past 2^32.  Encoded in a child process,
    so that the ~18 GB it holds on the device (the frame, the file twice, the encoder's scratch) is returned."""
    import torch
    free = torch.cuda.mem_get_info()[0]
    if free < 20 << 30:
        pytest.skip("needs 20 GB of free device memory; %.1f GB free" % (free / 2 ** 30))
    r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) +
                       [os.path.abspath(__file__), "past-4-gib"], capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["ok"], res
    print("past 4 GiB:", res)


def past_4_gib():
    """The child of test_file_past_4_gib: everything is checked on the device, the 4 GB file is never copied to
    the host."""
    import torch
    import rtrace_b200 as rt
    w, h, d2 = 16384, 16400, 32768
    chunks, n = (h + LINES - 1) // LINES, LINES * 4 * 4 * w
    free0 = torch.cuda.mem_get_info()[0]
    g = torch.Generator(device="cuda").manual_seed(17)
    frame = torch.empty((h, w, 4), dtype=torch.int32, device="cuda")
    frame[:1024 * LINES].random_(-2 ** 31, 2 ** 31 - 1, generator=g)
    frame[1024 * LINES:] = 0x07070707
    cap = rt.exr_bound(w, h)
    assert frame.numel() * 4 == 4299161600 and cap > 1 << 32
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    L, got = rt.lib(), rt.C.c_size_t()
    assert L.rt_encode_exr(frame.data_ptr(), 0, None, 0, w, h, out.data_ptr(), cap, rt.C.byref(got), None) == rt.RT_OK
    torch.cuda.synchronize()
    last = X.zlib_stream(X.predict(b"\x07" * n), d2)
    sizes = [n] * (chunks - 1) + [len(last)]
    head = len(X.header(w, h, 4))
    offs = head + 8 * chunks + np.concatenate(([0], np.cumsum([8 + s for s in sizes[:-1]])))
    assert offs[-1] > 1 << 32
    bad = []
    table = out[head:head + 8 * chunks].cpu().numpy().view("<u8")
    if not np.array_equal(table, offs):
        bad.append("offset table: first wrong entry %d" % int(np.flatnonzero(table != offs)[0]))
    idx = torch.from_numpy(offs).cuda()[:, None] + torch.arange(8, device="cuda")
    yz = out[idx].cpu().numpy().view("<i4")
    if not np.array_equal(yz, np.stack([np.arange(chunks) * LINES, sizes], 1)):
        bad.append("chunk y0/size: first wrong chunk %d" % int(np.flatnonzero((yz != np.stack(
            [np.arange(chunks) * LINES, sizes], 1)).any(1))[0]))
    perm = torch.tensor([3, 2, 1, 0], device="cuda")   # A B G R from {r, g, b, alpha}
    wrong = []
    for c in range(chunks - 1):
        want = frame[c * LINES:(c + 1) * LINES].index_select(2, perm).permute(0, 2, 1).contiguous().view(torch.uint8)
        o = int(offs[c]) + 8
        if not torch.equal(out[o:o + n], want.reshape(-1)):
            wrong.append(c)
    if wrong:
        bad.append("raw chunks differ: %s" % wrong[:10])
    o = int(offs[-1]) + 8
    if bytes(out[o:o + len(last)].cpu().numpy()) != last:
        bad.append("the last chunk's zlib stream differs")
    if got.value != cap - (n - len(last)):
        bad.append("length %d, want %d" % (got.value, cap - (n - len(last))))
    print(json.dumps({"ok": not bad, "problems": bad, "free_gb": round(free0 / 2 ** 30, 1),
                      "file_bytes": got.value, "last_chunk_offset": int(offs[-1]), "last_chunk_bytes": len(last)}))


if __name__ == "__main__":
    assert sys.argv[1:] == ["past-4-gib"], sys.argv
    past_4_gib()
