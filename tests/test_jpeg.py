"""JPEG output encoded on the GPU: rt_jpeg_bound, rt_encode_jpeg, rt_render_sweep_jpeg and `rtrace --format jpg`.

The layout is fixed (tests/_jpeg_ref.py, DESIGN.md "JPEG output"): the file is the one libjpeg-turbo writes through
Pillow for the same pixels with `quality=q, subsampling=2, restart_marker_rows=1`.  The reference encoder is checked
against Pillow on the CPU, and the device's files against both."""
import ctypes as C
import io
import json
import os
import subprocess

import numpy as np
import pytest

import _jpeg_ref as J

PIL = pytest.importorskip("PIL.Image")

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "target", "release", "rtrace")
GOLD = json.load(open(os.path.join(HERE, "golden", "rtrace_output_1024x768.json")))
DERIVED = json.load(open(os.path.join(HERE, "golden", "oracle_derived.json")))

QUALITIES = [1, 10, 50, 75, 90, 99, 100]
SIZES = [(1, 1), (1, 17), (7, 5), (8, 8), (15, 15), (16, 16), (17, 33), (31, 47), (64, 128)]  # (w, h)


def pillow(rgb, quality):
    f = io.BytesIO()
    PIL.fromarray(np.ascontiguousarray(rgb[..., :3])).save(f, "JPEG", quality=quality, subsampling=2,
                                                           restart_marker_rows=1)
    return f.getvalue()


def noise(h, w, seed=1):
    return np.random.default_rng(seed * 7919 + h * 131 + w).integers(0, 256, (h, w, 3)).astype(np.uint8)


def zrl_frame(h, w):
    """Grey 8x8 tiles built by an inverse DCT from two coefficients, at zig-zag positions 40 and 63: each luma block
    codes a run of 39 zeros (two ZRL codes) and then one of 22 (one ZRL code)."""
    k = np.arange(8)
    basis = np.sqrt(np.where(k == 0, 1.0, 2.0) / 8)[:, None] * np.cos(np.pi * (2 * k[None, :] + 1) * k[:, None] / 16)
    coef = np.zeros(64)
    coef[J.ZIGZAG[40]], coef[J.ZIGZAG[63]] = 300, -200
    tile = np.clip(np.round(basis.T @ coef.reshape(8, 8) @ basis + 128), 0, 255).astype(np.uint8)
    g = np.tile(tile, ((h + 7) // 8, (w + 7) // 8))[:h, :w]
    return np.repeat(g[:, :, None], 3, axis=2)


def gradient(h, w):
    yy, xx = np.mgrid[0:h, 0:w]
    return np.stack([(xx * 7) % 256, (yy * 5) % 256, ((xx + yy) * 3) % 256], -1).astype(np.uint8)


SYNTHETIC = {
    "noise": lambda h, w: noise(h, w),
    "constant": lambda h, w: np.full((h, w, 3), 77, np.uint8),
    "zrl": zrl_frame,
    "gradient": gradient,
}


# ---- the reference encoder against libjpeg-turbo ---------------------------------------------------------------
@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("kind", sorted(SYNTHETIC))
def test_reference_equals_pillow(w, h, kind):
    rgb = SYNTHETIC[kind](h, w)
    for q in QUALITIES:
        assert J.encode(rgb, q) == pillow(rgb, q), "%s %dx%d q%d" % (kind, w, h, q)


@pytest.mark.parametrize("w,h", [(8, 24), (24, 8), (40, 40), (2, 2), (18, 18), (300, 40)])
def test_reference_equals_pillow_at_even_heights_and_partial_mcus(w, h):
    """Heights that are even but not a multiple of 16 pad each component after downsampling, which differs from
    padding the pixels; widths past a multiple of 8 but not 16 make dummy luma blocks."""
    for kind in ("noise", "gradient"):
        rgb = SYNTHETIC[kind](h, w)
        for q in (50, 90, 100):
            assert J.encode(rgb, q) == pillow(rgb, q), "%s %dx%d q%d" % (kind, w, h, q)


def test_reference_drops_alpha():
    rgb = noise(20, 30)
    rgba = np.concatenate([rgb, np.full((20, 30, 1), 9, np.uint8)], axis=2)
    assert J.encode(rgba, 90) == J.encode(rgb, 90)


def test_cases_reach_zrl_and_stuffing():
    """The zrl frame codes runs of 16 zeros and more at every quality; noise at q100 makes 0xFF bytes in the
    entropy-coded data (stuffed)."""
    for q in QUALITIES:
        for b in J.coefficients(zrl_frame(16, 16), q).reshape(-1, 64)[:4]:
            z = np.flatnonzero(b[1:]) + 1
            assert z[0] > 16 and 63 in z, q
    data = J.encode(noise(64, 128), 100)[J.HEADER_BYTES:-2]
    assert data.count(b"\xff\x00") > 10


def test_reference_on_the_c1_frame(oracle_scene8):
    """C1 (`make image`) rendered by the CPU oracle, at q75 and q90 (83,595 bytes, as libjpeg-turbo writes it)."""
    img, _ = oracle_scene8.render(GOLD["width"], GOLD["height"], GOLD["spp"])
    rgb = np.ascontiguousarray(img[:, :, :3])
    for q in (75, 90):
        jpg = J.encode(rgb, q)
        assert jpg == pillow(rgb, q)
    assert len(J.encode(rgb, 90)) == 83595


def test_reference_decodes_in_pillow():
    rgb = gradient(37, 61)
    im = PIL.open(io.BytesIO(J.encode(rgb, 100)))
    assert im.size == (61, 37) and im.mode == "RGB"
    assert np.abs(np.asarray(im).astype(int) - rgb).mean() < 3


def bound_formula(w, h):
    """DESIGN.md "JPEG output": 629 header bytes, per MCU row 2 * (ceil(w/16) * 6 * 1660 / 8 + 1) + 2, then EOI."""
    return 629 + (h + 15) // 16 * (2 * ((w + 15) // 16 * 1245 + 1) + 2) + 2


def test_jpeg_bound_needs_no_device(rt):
    for (w, h) in [(1, 1), (2, 1), (17, 33), (1024, 768), (3840, 2160), (7680, 4320), (65535, 1), (1, 65535)]:
        assert rt.jpeg_bound(w, h) == bound_formula(w, h) == J.bound(w, h)
    for (h, w) in [(37, 50), (16, 16), (1, 1)]:
        assert rt.jpeg_bound(w, h) >= len(J.encode(noise(h, w), 100))
    for (w, h) in [(0, 1), (1, 0), (65536, 1), (1, 65536)]:
        with pytest.raises(rt.RtError) as e:
            rt.jpeg_bound(w, h)
        assert e.value.code == rt.RT_ERR_INVALID


# ---- command line without a device ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rtrace():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-s", "-C", ROOT, "rtrace"])
    return BIN


def run(rtrace, *args, cwd=None):
    return subprocess.run([rtrace] + list(args), capture_output=True, cwd=cwd, timeout=300)


def test_cli_jpg_needs_the_jpg_extension(rtrace, tmp_path):
    r = run(rtrace, "--format", "jpg", "picture.tga", cwd=str(tmp_path))
    assert r.returncode == 0
    assert r.stdout == b"Output file 'picture.tga' must have the jpg extension, e.g. picture.jpg\n"
    assert not list(tmp_path.iterdir())


@pytest.mark.parametrize("args,needle", [
    (["--format=jpg", "--buckets", "o.jpg"], b"--buckets"),
    (["--quality=90", "o.tga"], b"'--quality' can only be used with '--format jpg'"),
    (["--format=png", "--quality=90", "o.png"], b"'--quality' can only be used with '--format jpg'"),
    (["--format=jpg", "--quality=0", "o.jpg"], b"'0' is not a whole number in 1..100"),
    (["--format=jpg", "--quality=101", "o.jpg"], b"'101' is not a whole number in 1..100"),
    (["--format=jpg", "--quality", "x", "o.jpg"], b"'x' is not a whole number in 1..100"),
    (["--format=jpeg", "o.tga"], b"<ppm|tga|png|apng|pfm|exr|jpg>"),
])
def test_cli_jpg_usage_errors(rtrace, tmp_path, args, needle):
    r = run(rtrace, *args, cwd=str(tmp_path))
    assert r.returncode == 1 and needle in r.stderr, r.stderr
    assert not list(tmp_path.iterdir())


def test_cli_help_lists_jpg(rtrace):
    h = run(rtrace, "--help").stdout
    assert b"--format jpg" in h and b"--quality <Q>" in h and b".jpg" in h
    # the existing lines are unchanged
    for s in (b"<ppm|tga|png>", b"--fps <F>", b"--format exr", b"--format pfm", b"--preview <N>", b"--buckets",
              b"--samples-per-pixel", b"--num-cores", b"--aov"):
        assert s in h


# ---- on the GPU -------------------------------------------------------------------------------------------------
class DeviceFrame:
    """A frame rendered into device memory (rt_render_frame with a device output), and its bytes on the host."""

    def __init__(self, rt, scene, w, h, spp, camera=None):
        self.rt, self.w, self.h = rt, w, h
        self.ptr = rt.device_alloc(w * h * 4)
        rt.Renderer.render(rt.RenderOptions(w, h, spp), scene, camera=camera, out_ptr=self.ptr)
        self.rgba = np.empty((h, w, 4), np.uint8)
        rt.memcpy(self.rgba.ctypes.data, self.ptr, self.rgba.nbytes)

    def encode(self, quality=90):
        return self.rt.encode_jpeg(self.ptr, self.w, self.h, quality)

    def close(self):
        self.rt.device_free(self.ptr)


def on_device(rt, rgba, quality):
    rgba = np.ascontiguousarray(rgba)
    h, w, _ = rgba.shape
    ptr = rt.device_alloc(rgba.nbytes)
    try:
        rt.memcpy(ptr, rgba.ctypes.data, rgba.nbytes)
        return rt.encode_jpeg(ptr, w, h, quality)
    finally:
        rt.device_free(ptr)


def with_alpha(rgb, seed=3):
    h, w, _ = rgb.shape
    alpha = np.random.default_rng(seed).integers(0, 256, (h, w, 1)).astype(np.uint8)
    return np.concatenate([rgb, alpha], axis=2)


FIXTURE_CASES = [c for c in DERIVED["cases"] if (c["width"], c["height"], c["spp"], c["level"]) in
                 [(1024, 768, 4, 8), (3840, 2160, 1, 8), (3840, 2160, 4, 9), (7680, 4320, 4, 9)]]


@pytest.mark.gpu
@pytest.mark.parametrize("case", FIXTURE_CASES,
                         ids=lambda c: "%dx%d_spp%d_L%d" % (c["width"], c["height"], c["spp"], c["level"]))
def test_encode_fixture_frames(rt, case):
    """C1, C2, C3 and C4: the device frame is the oracle's, and its JPEG at q 1, 75, 90 and 100 is Pillow's file
    (and the reference encoder's at 1024x768)."""
    import hashlib
    scene = rt.Scene(level=case["level"])
    f = DeviceFrame(rt, scene, case["width"], case["height"], case["spp"])
    try:
        assert hashlib.sha256(f.rgba.tobytes()).hexdigest() == case["rgba_sha256"]
        for q in (1, 75, 90, 100):
            jpg = f.encode(q)
            assert jpg == pillow(f.rgba, q), "q%d" % q
            if case["width"] == 1024:
                assert jpg == J.encode(f.rgba, q)
                if q == 90:
                    assert len(jpg) == 83595
    finally:
        f.close()


@pytest.mark.gpu
def test_encode_c5_orbit_frames(rt):
    import hashlib
    cases = DERIVED["c5_cases"]
    scene = rt.Scene(level=cases[0]["level"])
    for c in cases:
        f = DeviceFrame(rt, scene, c["width"], c["height"], c["spp"], camera=rt.orbit_camera(c["frame"], c["n_frames"]))
        try:
            assert hashlib.sha256(f.rgba.tobytes()).hexdigest() == c["rgba_sha256"], "orbit frame %d" % c["frame"]
            assert f.encode(90) == pillow(f.rgba, 90), "orbit frame %d" % c["frame"]
        finally:
            f.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,spp", [(1, 1, 1), (17, 33, 2), (8, 8, 1), (24, 8, 3), (300, 16, 4), (65535, 1, 1),
                                     (1, 40, 1), (203, 45, 2)])
def test_encode_odd_sizes(rt, gpu_scene8, oracle_scene8, w, h, spp):
    f = DeviceFrame(rt, gpu_scene8, w, h, spp)
    try:
        ref, _ = oracle_scene8.render(w, h, spp)
        assert np.array_equal(f.rgba, ref)
        for q in (1, 75, 90, 100):
            assert f.encode(q) == J.encode(f.rgba, q), "q%d" % q
    finally:
        f.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pad_px", [13, 4])
def test_encode_pitched_input(rt, gpu_scene8, pad_px):
    """Row pitches wider than the row: one not a multiple of 16 bytes (byte loads) and one that is (16-byte loads)."""
    w, h, spp = 203, 45, 2
    pitch = (w + pad_px) * 4
    ptr = rt.device_alloc(pitch * h)
    try:
        rt.Renderer.render_rows(rt.RenderOptions(w, h, spp), gpu_scene8, out_ptr=ptr, pitch=pitch, row_count=h)
        padded = np.empty((h, pitch), np.uint8)
        rt.memcpy(padded.ctypes.data, ptr, padded.nbytes)
        rgb = np.ascontiguousarray(padded[:, :w * 4].reshape(h, w, 4)[:, :, :3])
        assert rt.encode_jpeg(ptr, w, h, 90, pitch=pitch) == J.encode(rgb, 90)
    finally:
        rt.device_free(ptr)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(SYNTHETIC))
def test_encode_synthetic_frames(rt, kind):
    """Noise (the largest codes, many stuffed 0xFF bytes), constant frames (EOB-only blocks), the zrl frame (ZRL
    runs) and a gradient, from RGBA with random alpha, which is dropped."""
    for (w, h) in [(77, 33), (64, 128), (16, 16), (31, 47)]:
        rgb = SYNTHETIC[kind](h, w)
        for q in (1, 75, 90, 100):
            assert on_device(rt, with_alpha(rgb), q) == J.encode(rgb, q), "%dx%d q%d" % (w, h, q)


@pytest.mark.gpu
def test_encode_noise_4k_equals_pillow(rt):
    rgb = noise(2160, 3840)
    assert on_device(rt, with_alpha(rgb), 100) == pillow(rgb, 100)


@pytest.mark.gpu
def test_encode_errors(rt, gpu_scene8):
    L = rt.lib()
    f = DeviceFrame(rt, gpu_scene8, 64, 48, 1)
    try:
        full = f.encode(90)
        n = C.c_size_t()
        short = C.create_string_buffer(len(full) - 1)
        rc = L.rt_encode_jpeg(C.c_void_p(f.ptr), 64, 48, 0, 90, short, len(full) - 1, C.byref(n), None)
        assert rc == rt.RT_ERR_BUFFER and n.value == len(full)
        host = np.zeros((48, 64, 4), np.uint8)
        out = C.create_string_buffer(len(full))
        assert L.rt_encode_jpeg(C.c_void_p(host.ctypes.data), 64, 48, 0, 90, out, len(full), C.byref(n), None) == rt.RT_ERR_INVALID
        assert L.rt_encode_jpeg(C.c_void_p(f.ptr), 0, 48, 0, 90, out, len(full), C.byref(n), None) == rt.RT_ERR_INVALID
        assert L.rt_encode_jpeg(C.c_void_p(f.ptr), 64, 0, 0, 90, out, len(full), C.byref(n), None) == rt.RT_ERR_INVALID
        for q in (0, 101, -5):
            assert L.rt_encode_jpeg(C.c_void_p(f.ptr), 64, 48, 0, q, out, len(full), C.byref(n), None) == rt.RT_ERR_INVALID
        assert L.rt_encode_jpeg(C.c_void_p(f.ptr), 64, 48, 0, 90, out, len(full), C.byref(n), None) == rt.RT_OK
        assert out.raw[:n.value] == full
        # into device memory: the same bytes
        dptr = rt.device_alloc(len(full))
        try:
            assert L.rt_encode_jpeg(C.c_void_p(f.ptr), 64, 48, 0, 90, C.c_void_p(dptr), len(full), C.byref(n), None) == rt.RT_OK
            back = np.empty(n.value, np.uint8)
            rt.memcpy(back.ctypes.data, dptr, n.value)
            assert back.tobytes() == full
        finally:
            rt.device_free(dptr)
    finally:
        f.close()


def check_jpeg_sweep(rt, scenes, w, h, spp, n, quality):
    cams = [rt.orbit_camera(k, 24) for k in range(n)]
    order, files = [], {}
    st = rt.Renderer.render_sweep_jpeg(rt.RenderOptions(w, h, spp), scenes, n, cameras=cams, quality=quality,
                                       on_frame=lambda k, b: (order.append(k), files.__setitem__(k, b)))
    assert order == list(range(n)) and st.gpus == len(scenes)
    for k in range(n):
        f = DeviceFrame(rt, scenes[0], w, h, spp, camera=cams[k])
        try:
            assert files[k] == f.encode(quality), "frame %d" % k
            assert files[k] == J.encode(f.rgba, quality), "frame %d" % k
        finally:
            f.close()


@pytest.mark.gpu
def test_sweep_jpeg_single_gpu(rt, gpu_scene8):
    check_jpeg_sweep(rt, [gpu_scene8], 320, 200, 2, 7, 90)
    check_jpeg_sweep(rt, [gpu_scene8], 97, 41, 1, 3, 75)
    with pytest.raises(rt.RtError) as e:
        rt.Renderer.render_sweep_jpeg(rt.RenderOptions(32, 32, 1), [gpu_scene8], 2, quality=0)
    assert e.value.code == rt.RT_ERR_INVALID


@pytest.mark.gpu
def test_sweep_jpeg_two_gpus(rt):
    if rt.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    scenes = []
    for g in range(2):
        rt.set_device(g)
        scenes.append(rt.Scene())
    rt.set_device(0)
    check_jpeg_sweep(rt, scenes, 320, 200, 2, 7, 90)


@pytest.mark.gpu
def test_cli_jpg_make_image(rtrace, oracle_scene8, tmp_path):
    r = run(rtrace, "--format", "jpg", "--samples-per-pixel=4", "--width=1024", "--height=768", "out.jpg",
            cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr
    jpg = (tmp_path / "out.jpg").read_bytes()
    img, _ = oracle_scene8.render(1024, 768, 4)
    assert jpg == pillow(img, 90)
    s = run(rtrace, "--format=jpg", "--samples-per-pixel=4", "--width=1024", "--height=768", "-")
    assert s.returncode == 0 and s.stdout == jpg
    t = run(rtrace, "--format=jpg", "--quality=75", "--samples-per-pixel=4", "--width=1024", "--height=768", "-")
    assert t.returncode == 0 and t.stdout == pillow(img, 75) and t.stdout != jpg


@pytest.mark.gpu
def test_cli_jpg_frames_and_preview(rtrace, tmp_path):
    w, h = 160, 96
    a = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "a.tga", cwd=str(tmp_path))
    b = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "--format=jpg", "b.jpg", cwd=str(tmp_path))
    c = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "--format=jpg", "-")
    assert a.returncode == 0 and b.returncode == 0 and c.returncode == 0, b.stderr
    hdr = len(b"P6\n160 96\n255\n")
    files = []
    for k in range(3):
        body = np.frombuffer((tmp_path / ("a.%04d.tga" % k)).read_bytes()[hdr:], np.uint8).reshape(h, w, 3)
        files.append((tmp_path / ("b.%04d.jpg" % k)).read_bytes())
        assert files[-1] == J.encode(body, 90), k
    assert c.stdout == b"".join(files)
    p = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--preview=4", "--format=jpg", "-")
    q = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--preview=4", "-")
    assert p.returncode == 0 and p.stdout == J.encode(np.frombuffer(q.stdout[hdr:], np.uint8).reshape(h, w, 3), 90)


@pytest.mark.gpu
def test_cli_jpg_two_gpus(rtrace, tmp_path):
    import rtrace_b200 as rt
    if rt.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    one = run(rtrace, "--format=jpg", "--gpus=1", "--width=640", "--height=360", "-")
    two = run(rtrace, "--format=jpg", "--gpus=2", "--width=640", "--height=360", "-")
    assert one.returncode == 0 and two.returncode == 0 and one.stdout == two.stdout
