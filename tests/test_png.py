"""PNG output encoded on the GPU: rt_png_bound, rt_encode_png, rt_render_sweep_png and `rtrace --format png`.

The layout is fixed (tests/_png_ref.py, DESIGN.md "PNG output"), so the device's file is compared with the
reference encoder byte for byte, and every file is decoded through the chunk walker (signature, IHDR, every CRC,
zlib's Adler-32 check) back to the frame's RGB."""
import ctypes as C
import hashlib
import json
import os
import struct
import subprocess

import numpy as np
import pytest

import _png_ref as P

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "target", "release", "rtrace")
GOLD = json.load(open(os.path.join(HERE, "golden", "rtrace_output_1024x768.json")))
DERIVED = json.load(open(os.path.join(HERE, "golden", "oracle_derived.json")))
REF_ROWS = os.path.join(HERE, "golden", "rtrace_output_1024x768_rows.npz")


def check_file(png, rgb):
    """The file walks, decodes to `rgb` and has the fixed layout: header chunks, one IDAT per 16-row band, the
    final IDAT and IEND."""
    h, w, _ = rgb.shape
    cs = P.chunks(png)
    assert [t for t, _ in cs] == [b"IHDR"] + [b"IDAT"] * (2 + (h + 15) // 16) + [b"IEND"]
    assert cs[1][1] == b"\x78\x01" and cs[-2][1][:2] == b"\x03\x00"
    assert np.array_equal(P.decode(png), rgb)
    assert len(png) <= P.bound(w, h)


def one_colour_row(w, rgb=(7, 7, 7)):
    return np.tile(np.array(rgb, np.uint8), (1, w, 1))


def row_of(first, rest, n):
    return np.array([[first] + [rest] * n], np.uint8)


NOISE = np.random.default_rng(1234).integers(0, 256, (37, 50, 3)).astype(np.uint8)

REFERENCE_CASES = {
    "1x1": np.array([[[200, 10, 144]]], np.uint8),
    "2x1": np.array([[[1, 2, 3], [1, 2, 3]]], np.uint8),
    "run258_mod0": one_colour_row(87),              # R = 3W - 3 = 258
    "run261_mod3": one_colour_row(88),              # 258 + a match of 3
    "run259_mod1": row_of((1, 2, 3), (9, 8, 3), 87),  # the blue run is one longer: 258 + one literal
    "run260_mod2": row_of((1, 2, 3), (9, 2, 3), 87),  # green and blue: 258 + two literals
    "run_long": one_colour_row(1000, (150, 150, 150)),
    "one_colour_frame": np.full((40, 70, 3), 200, np.uint8),
    "noise": NOISE,
    "h15": NOISE[:15],
    "h16": np.concatenate([NOISE, NOISE])[:16],
    "h17": np.concatenate([NOISE, NOISE])[:17],
}


@pytest.mark.parametrize("name", sorted(REFERENCE_CASES))
def test_reference_encoder_round_trips(name):
    rgb = REFERENCE_CASES[name]
    png = P.encode(rgb)
    check_file(png, rgb)
    w, h, depth, ctype, comp, filt, interlace = struct.unpack(">IIBBBBB", P.chunks(png)[0][1])
    assert (w, h, depth, ctype, comp, filt, interlace) == (rgb.shape[1], rgb.shape[0], 8, 2, 0, 0, 0)


def test_reference_encoder_run_rule():
    """The closed-form parse: a run of 258 is one 13-bit match; 259 and 260 add one and two literals; 261 adds a
    match of 3 -- so the piece sizes step exactly as the token lengths say."""
    def piece_bits(rgb):
        bw = P.Bits()
        P.encode_row(bw, b"\x00" + rgb[0].tobytes())
        return len(bw.out)
    base = 3 + 8 + 3 * 8 + 7 + 3   # header, filter byte, first pixel (all < 144), end-of-block, stored header
    assert piece_bits(one_colour_row(87)) == (base + 13 + 7) // 8 + 4
    assert piece_bits(one_colour_row(88)) == (base + 13 + 12 + 7) // 8 + 4


def test_reference_encoder_on_the_c1_frame(oracle_scene8):
    """C1 (`make image`) rendered by the CPU oracle: 562,214 bytes, decoding to the reference image's RGB."""
    img, _ = oracle_scene8.render(GOLD["width"], GOLD["height"], GOLD["spp"])
    rgb = np.ascontiguousarray(img[:, :, :3])
    png = P.encode(rgb)
    assert len(png) == 562214
    check_file(png, rgb)
    dec = P.decode(png)
    assert hashlib.sha256(dec.tobytes()).hexdigest() == GOLD["rgb_sha256"]
    ref = np.load(REF_ROWS)
    assert np.array_equal(dec[ref["rows"].astype(np.int64)], ref["rgb"])


def test_png_bound_needs_no_device(rt):
    for (w, h) in [(1, 1), (2, 1), (17, 33), (1024, 768), (3840, 2160), (7680, 4320), (65535, 1), (1, 65535)]:
        assert rt.png_bound(w, h) == P.bound(w, h)
    for rgb in (NOISE, REFERENCE_CASES["1x1"], np.full((17, 3, 3), 255, np.uint8)):
        assert rt.png_bound(rgb.shape[1], rgb.shape[0]) >= len(P.encode(rgb))
    for (w, h) in [(0, 1), (1, 0), (65536, 1)]:
        with pytest.raises(rt.RtError) as e:
            rt.png_bound(w, h)
        assert e.value.code == rt.RT_ERR_INVALID


# ---- command line without a device ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rtrace():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-s", "-C", ROOT, "rtrace"])
    return BIN


def run(rtrace, *args, cwd=None):
    return subprocess.run([rtrace] + list(args), capture_output=True, cwd=cwd, timeout=300)


def test_cli_png_needs_the_png_extension(rtrace, tmp_path):
    r = run(rtrace, "--format", "png", "picture.tga", cwd=str(tmp_path))
    assert r.returncode == 0
    assert r.stdout == b"Output file 'picture.tga' must have the png extension, e.g. picture.png\n"
    assert not list(tmp_path.iterdir())


def test_cli_png_rejects_buckets_and_is_listed(rtrace, tmp_path):
    r = run(rtrace, "--format=png", "--buckets", "o.png", cwd=str(tmp_path))
    assert r.returncode == 1 and b"--buckets" in r.stderr
    assert b"<ppm|tga|png>" in run(rtrace, "--help").stdout


# ---- on the GPU -------------------------------------------------------------------------------------------------
class DeviceFrame:
    """A frame rendered into device memory (rt_render_frame with a device output), and its bytes on the host."""

    def __init__(self, rt, scene, w, h, spp, camera=None):
        self.rt, self.w, self.h = rt, w, h
        self.ptr = rt.device_alloc(w * h * 4)
        _, self.stats = rt.Renderer.render(rt.RenderOptions(w, h, spp), scene, camera=camera, out_ptr=self.ptr,
                                           want_stats=True)
        self.rgba = np.empty((h, w, 4), np.uint8)
        rt.memcpy(self.rgba.ctypes.data, self.ptr, self.rgba.nbytes)
        self.rgb = np.ascontiguousarray(self.rgba[:, :, :3])

    def encode(self):
        return self.rt.encode_png(self.ptr, self.w, self.h)

    def close(self):
        self.rt.device_free(self.ptr)


def check_device_encode(frame, ppm_sha256=None, rgb_sha256=None):
    png = frame.encode()
    assert png == P.encode(frame.rgb), "device file differs from the reference encoder"
    check_file(png, frame.rgb)
    dec = P.decode(png)
    if ppm_sha256:
        ppm = b"P6\n%d %d\n255\n" % (frame.w, frame.h) + dec.tobytes()
        assert hashlib.sha256(ppm).hexdigest() == ppm_sha256
    if rgb_sha256:
        assert hashlib.sha256(dec.tobytes()).hexdigest() == rgb_sha256
    return png


FIXTURE_CASES = [c for c in DERIVED["cases"] if (c["width"], c["height"], c["spp"], c["level"]) in
                 [(1024, 768, 4, 8), (3840, 2160, 1, 8), (3840, 2160, 4, 9), (7680, 4320, 4, 9), (64, 128, 2, 8)]]


@pytest.mark.gpu
@pytest.mark.parametrize("case", FIXTURE_CASES,
                         ids=lambda c: "%dx%d_spp%d_L%d" % (c["width"], c["height"], c["spp"], c["level"]))
def test_encode_matches_reference_on_fixture_frames(rt, case):
    """C1, C2 at level 8, C3, C4 and 64x128: the rendered device frame is the oracle's (rgba_sha256), and its PNG
    is the reference encoder's file byte for byte and decodes to the P6 body of the fixture."""
    scene = rt.Scene(level=case["level"])
    f = DeviceFrame(rt, scene, case["width"], case["height"], case["spp"])
    try:
        assert hashlib.sha256(f.rgba.tobytes()).hexdigest() == case["rgba_sha256"]
        if case["width"] * case["height"] >= 1024 * 768:
            assert f.stats.variant_used in (rt.VARIANT_TILE, rt.VARIANT_PHASED)
        png = check_device_encode(f, ppm_sha256=case["ppm_sha256"])
        if (case["width"], case["height"], case["spp"], case["level"]) == (1024, 768, 4, 8):
            assert len(png) == 562214
            assert hashlib.sha256(P.decode(png).tobytes()).hexdigest() == GOLD["rgb_sha256"]
    finally:
        f.close()


@pytest.mark.gpu
def test_encode_matches_reference_on_c5_orbit_frames(rt):
    cases = DERIVED["c5_cases"]
    scene = rt.Scene(level=cases[0]["level"])
    for c in cases:
        f = DeviceFrame(rt, scene, c["width"], c["height"], c["spp"], camera=rt.orbit_camera(c["frame"], c["n_frames"]))
        try:
            assert hashlib.sha256(f.rgba.tobytes()).hexdigest() == c["rgba_sha256"], "orbit frame %d" % c["frame"]
            check_device_encode(f, rgb_sha256=c["rgb_sha256"])
        finally:
            f.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,spp", [(1, 1, 1), (17, 33, 2), (65535, 1, 1), (1, 40, 1), (300, 16, 3)])
def test_encode_odd_sizes(rt, gpu_scene8, oracle_scene8, w, h, spp):
    f = DeviceFrame(rt, gpu_scene8, w, h, spp)
    try:
        ref, _ = oracle_scene8.render(w, h, spp)
        assert np.array_equal(f.rgba, ref)
        check_device_encode(f)
    finally:
        f.close()


@pytest.mark.gpu
def test_encode_pitched_input_and_synthetic_frames(rt, gpu_scene8):
    """A frame with a row pitch wider than the row, and frames no renderer makes: noise (every literal, the
    9-bit range), one colour (runs across the 258 cap), a row of runs of every remainder."""
    w, h, spp = 203, 45, 2
    pitch = (w + 13) * 4
    ptr = rt.device_alloc(pitch * h)
    try:
        rt.Renderer.render_rows(rt.RenderOptions(w, h, spp), gpu_scene8, out_ptr=ptr, pitch=pitch, row_count=h)
        padded = np.empty((h, pitch), np.uint8)
        rt.memcpy(padded.ctypes.data, ptr, padded.nbytes)
        rgb = np.ascontiguousarray(padded[:, :w * 4].reshape(h, w, 4)[:, :, :3])
        assert rt.encode_png(ptr, w, h, pitch=pitch) == P.encode(rgb)
    finally:
        rt.device_free(ptr)
    rng = np.random.default_rng(7)
    runs = np.repeat(rng.integers(0, 256, (50, 4)), rng.integers(1, 400, 50), axis=0)[None].astype(np.uint8)
    for rgba in (rng.integers(0, 256, (33, 77, 4)).astype(np.uint8), np.full((20, 900, 4), 160, np.uint8), runs):
        rgba = np.ascontiguousarray(rgba)
        hh, ww, _ = rgba.shape
        ptr = rt.device_alloc(rgba.nbytes)
        try:
            rt.memcpy(ptr, rgba.ctypes.data, rgba.nbytes)
            png = rt.encode_png(ptr, ww, hh)
            assert png == P.encode(rgba[:, :, :3])
            check_file(png, np.ascontiguousarray(rgba[:, :, :3]))
        finally:
            rt.device_free(ptr)


def lane_rows():
    """32 rows, row L with one run of 258 repeated bytes (87 pixels of one colour) starting at raw-row byte p with
    p = L mod 32: the lane of the 32-byte step where the run starts.  The other pixels repeat no byte 3 back."""
    rows = []
    for lane in range(32):
        x0 = (lane - 4) * 11 % 32                      # the run starts at byte 1 + 3 * (x0 + 1); 3 * 11 = 1 mod 32
        px = [[(7 * k + c) % 97 for c in range(3)] for k in range(120)]
        px[x0:x0 + 87] = [[200, 201, 202]] * 87
        rows.append(px)
    return np.array(rows, np.uint8)


DEVICE_CASES = dict(REFERENCE_CASES, run258_lanes=lane_rows())


def test_lane_rows_start_a_258_run_at_every_lane():
    starts = set()
    for row in lane_rows():
        a = np.frombuffer(b"\x00" + row.tobytes(), np.uint8)
        eq = np.flatnonzero(a[4:] == a[1:-3]) + 4
        assert len(eq) == 258 and eq[-1] - eq[0] == 257
        starts.add(int(eq[0]) % 32)
    assert starts == set(range(32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(DEVICE_CASES))
def test_encode_reference_cases_on_the_device(rt, name):
    """The crafted cases (runs of every remainder mod 258, band heights 15/16/17, runs starting at every lane)
    encoded on the device from RGBA with random alpha, which must be dropped."""
    rgb = DEVICE_CASES[name]
    h, w, _ = rgb.shape
    alpha = np.random.default_rng(len(name) * 131 + h).integers(0, 256, (h, w, 1)).astype(np.uint8)
    rgba = np.ascontiguousarray(np.concatenate([rgb, alpha], axis=2))
    ptr = rt.device_alloc(rgba.nbytes)
    try:
        rt.memcpy(ptr, rgba.ctypes.data, rgba.nbytes)
        png = rt.encode_png(ptr, w, h)
    finally:
        rt.device_free(ptr)
    assert png == P.encode(rgb)
    check_file(png, rgb)


@pytest.mark.gpu
def test_encode_errors(rt, gpu_scene8):
    L = rt.lib()
    f = DeviceFrame(rt, gpu_scene8, 64, 48, 1)
    try:
        full = f.encode()
        n = C.c_size_t()
        short = C.create_string_buffer(len(full) - 1)
        rc = L.rt_encode_png(C.c_void_p(f.ptr), 64, 48, 0, short, len(full) - 1, C.byref(n), None)
        assert rc == rt.RT_ERR_BUFFER and n.value == len(full)
        host = np.zeros((48, 64, 4), np.uint8)
        out = C.create_string_buffer(len(full))
        assert L.rt_encode_png(C.c_void_p(host.ctypes.data), 64, 48, 0, out, len(full), C.byref(n), None) == rt.RT_ERR_INVALID
        assert L.rt_encode_png(C.c_void_p(f.ptr), 0, 48, 0, out, len(full), C.byref(n), None) == rt.RT_ERR_INVALID
        assert L.rt_encode_png(C.c_void_p(f.ptr), 64, 48, 0, out, len(full), C.byref(n), None) == rt.RT_OK
        assert out.raw[:n.value] == full
    finally:
        f.close()


def check_png_sweep(rt, scenes, w, h, spp, n):
    cams = [rt.orbit_camera(k, 24) for k in range(n)]
    order, files = [], {}
    st = rt.Renderer.render_sweep_png(rt.RenderOptions(w, h, spp), scenes, n, cameras=cams,
                                      on_frame=lambda k, b: (order.append(k), files.__setitem__(k, b)))
    assert order == list(range(n)) and st.gpus == len(scenes)
    rgbs = {}
    rt.Renderer.render_sweep_multi(rt.RenderOptions(w, h, spp), scenes, n, cameras=cams, rgb=True,
                                   on_frame=lambda k, a: rgbs.__setitem__(k, a.copy()))
    for k in range(n):
        f = DeviceFrame(rt, scenes[0], w, h, spp, camera=cams[k])
        try:
            assert files[k] == f.encode(), "frame %d" % k
        finally:
            f.close()
        assert np.array_equal(P.decode(files[k]), rgbs[k]), "frame %d" % k


@pytest.mark.gpu
def test_sweep_png_single_gpu(rt, gpu_scene8):
    check_png_sweep(rt, [gpu_scene8], 320, 200, 2, 7)


@pytest.mark.gpu
def test_sweep_png_two_gpus(rt):
    if rt.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    scenes = []
    for g in range(2):
        rt.set_device(g)
        scenes.append(rt.Scene())
    rt.set_device(0)
    check_png_sweep(rt, scenes, 320, 200, 2, 7)


@pytest.mark.gpu
def test_cli_png_make_image_is_the_reference_image(rtrace, tmp_path):
    r = run(rtrace, "--format", "png", "--samples-per-pixel=4", "--width=1024", "--height=768", "out.png",
            cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr
    png = (tmp_path / "out.png").read_bytes()
    assert len(png) == 562214
    assert hashlib.sha256(P.decode(png).tobytes()).hexdigest() == GOLD["rgb_sha256"]
    s = run(rtrace, "--format=png", "--samples-per-pixel=4", "--width=1024", "--height=768", "-")
    assert s.returncode == 0 and s.stdout == png


@pytest.mark.gpu
def test_cli_png_frames_hold_the_p6_pixels(rtrace, tmp_path):
    w, h = 160, 96
    a = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "a.tga", cwd=str(tmp_path))
    b = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "--format=png", "b.png", cwd=str(tmp_path))
    assert a.returncode == 0 and b.returncode == 0, b.stderr
    hdr = len(b"P6\n160 96\n255\n")
    for k in range(3):
        body = (tmp_path / ("a.%04d.tga" % k)).read_bytes()[hdr:]
        assert P.decode((tmp_path / ("b.%04d.png" % k)).read_bytes()).tobytes() == body, k
    # a preview goes through the same encoder
    p = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--preview=4", "--format=png", "-")
    q = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--preview=4", "-")
    assert p.returncode == 0 and P.decode(p.stdout).tobytes() == q.stdout[hdr:]
