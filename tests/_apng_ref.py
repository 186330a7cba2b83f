"""Reference writer and chunk walker of the animated PNG layout rt_encode_apng_frame writes.  TEST INFRASTRUCTURE.

The layout (DESIGN.md "Animated PNG") is built on _png_ref.encode: every frame's zlib chunks are exactly the ones
of its stand-alone PNG (C = bands + 2 of them).  Frame 0 is the signature, IHDR, acTL, fcTL 0 and its IDAT chunks;
frame f >= 1 is fcTL s_f and its chunks as fdAT, chunk k numbered s_f + 1 + k, where s_f = 1 + (f - 1)(C + 1); the
last frame ends with IEND.  `payloads` returns each frame's piece; the file is their concatenation.
"""
import struct

import numpy as np

import _png_ref as P


def chunk_count(h):
    return (h + P.BAND - 1) // P.BAND + 2


def fctl_seq(f, h):
    return 0 if f == 0 else 1 + (f - 1) * (chunk_count(h) + 1)


def payloads(frames, delay_num=1, delay_den=24):
    """One byte string per frame of (h, w, 3) uint8 frames, in order."""
    return payloads_of_pngs([P.encode(rgb) for rgb in frames], delay_num, delay_den)


def payloads_of_pngs(pngs, delay_num=1, delay_den=24):
    """The same from the frames' stand-alone PNG files in the layout of _png_ref.encode."""
    n = len(pngs)
    out = []
    for f, png in enumerate(pngs):
        cs = P.chunks(png)
        w, h = struct.unpack(">II", cs[0][1][:8])
        zchunks = [d for t, d in cs if t == b"IDAT"]
        assert len(zchunks) == chunk_count(h)
        s = fctl_seq(f, h)
        parts = []
        if f == 0:
            parts += [P.SIGNATURE, P.chunk(b"IHDR", cs[0][1]), P.chunk(b"acTL", struct.pack(">II", n, 0))]
        parts.append(P.chunk(b"fcTL", struct.pack(">IIIIIHHBB", s, w, h, 0, 0, delay_num, delay_den, 0, 0)))
        for k, d in enumerate(zchunks):
            parts.append(P.chunk(b"IDAT", d) if f == 0 else P.chunk(b"fdAT", struct.pack(">I", s + 1 + k) + d))
        if f == n - 1:
            parts.append(P.chunk(b"IEND", b""))
        out.append(b"".join(parts))
    return out


def encode(frames, delay_num=1, delay_den=24):
    return b"".join(payloads(frames, delay_num, delay_den))


def size_identity(png_sizes, h):
    """The animation's length from its frames' stand-alone PNG lengths: the signature, IHDR and IEND (45 bytes) once
    instead of n times, one acTL (20), an fcTL (38) per frame and a sequence number per chunk of every later frame."""
    n = len(png_sizes)
    return sum(png_sizes) - 45 * (n - 1) + 20 + 38 * n + 4 * chunk_count(h) * (n - 1)


def frame_bound(png_bound, h):
    """rt_apng_bound's arithmetic: the PNG bound, acTL, fcTL and a sequence number per chunk."""
    return png_bound + 58 + 4 * chunk_count(h)


def walk(apng):
    """Walk an animated PNG's chunks (signature, lengths and CRCs by _png_ref.chunks), check that the sequence
    numbers of fcTL and fdAT run 0, 1, 2, ... without gaps and that every frame has its fcTL and data; returns
    (chunks, acTL (num_frames, num_plays), [fcTL fields per frame])."""
    cs = P.chunks(apng)
    assert cs[0][0] == b"IHDR" and cs[1][0] == b"acTL" and cs[2][0] == b"fcTL" and cs[-1] == (b"IEND", b"")
    actl = struct.unpack(">II", cs[1][1])
    seq, fctls, data_since_fctl = 0, [], True
    for t, d in cs:
        if t in (b"fcTL", b"fdAT"):
            assert struct.unpack(">I", d[:4])[0] == seq, "sequence number %d expected in %r" % (seq, t)
            seq += 1
        if t == b"fcTL":
            assert data_since_fctl, "fcTL without frame data"
            fctls.append(struct.unpack(">IIIIIHHBB", d))
            data_since_fctl = False
        elif t in (b"IDAT", b"fdAT"):
            assert t == (b"IDAT" if len(fctls) == 1 else b"fdAT"), "%r in frame %d" % (t, len(fctls) - 1)
            data_since_fctl = True
    assert data_since_fctl and actl[0] == len(fctls)
    return cs, actl, fctls


def strip_animation(apng):
    """The file without acTL, fcTL and fdAT: the plain PNG of frame 0."""
    cs = P.chunks(apng)
    return P.SIGNATURE + b"".join(P.chunk(t, d) for t, d in cs if t in (b"IHDR", b"IDAT", b"IEND"))


def decode_frames(apng):
    """Every frame as (h, w, 3) uint8 through this project's own decoder (IHDR + each frame's zlib stream)."""
    cs, _, _ = walk(apng)
    ihdr = P.chunk(b"IHDR", cs[0][1])
    frames, cur = [], None
    for t, d in cs:
        if t == b"fcTL":
            cur = []
            frames.append(cur)
        elif t in (b"IDAT", b"fdAT"):
            cur.append(d if t == b"IDAT" else d[4:])
    return [P.decode(P.SIGNATURE + ihdr + b"".join(P.chunk(b"IDAT", d) for d in fr) + P.chunk(b"IEND", b""))
            for fr in frames]


def pillow_frames(apng):
    """(frames as (h, w, 3) uint8, durations in ms) decoded by Pillow, an independent APNG reader."""
    import io
    from PIL import Image
    im = Image.open(io.BytesIO(apng))
    frames, durations = [], []
    for k in range(getattr(im, "n_frames", 1)):
        im.seek(k)
        frames.append(np.asarray(im.convert("RGB")).copy())
        durations.append(im.info.get("duration"))
    return frames, durations
