"""Animated PNG of the orbit sweep, encoded on the GPU: rt_apng_bound, rt_encode_apng_frame, rt_render_sweep_apng
and `rtrace --format apng`.

The layout is fixed (tests/_apng_ref.py, DESIGN.md "Animated PNG"), so every payload the device writes is compared
byte for byte with the reference writer's, and files are read back by the chunk walker (CRCs, sequence numbers),
by the project's own decoder and by Pillow."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import _apng_ref as A
import _png_ref as P

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "target", "release", "rtrace")
GOLD = json.load(open(os.path.join(HERE, "golden", "rtrace_output_1024x768.json")))
DERIVED = json.load(open(os.path.join(HERE, "golden", "oracle_derived.json")))


def check_animation(apng, frames, delay_num=1, delay_den=24):
    """Walks with every CRC and sequence number right, decodes (ours and Pillow's) to `frames` with their
    duration, is the PNG of frame 0 without the animation chunks, and has the length the size identity gives."""
    h, w, _ = frames[0].shape
    _, actl, fctls = A.walk(apng)
    assert actl == (len(frames), 0)
    assert all(fc[1:] == (w, h, 0, 0, delay_num, delay_den, 0, 0) for fc in fctls)
    for k, (ours, ref) in enumerate(zip(A.decode_frames(apng), frames)):
        assert np.array_equal(ours, ref), "frame %d" % k
    pil, durations = A.pillow_frames(apng)
    assert len(pil) == len(frames)
    for k, (img, ref) in enumerate(zip(pil, frames)):
        assert np.array_equal(img, ref), "Pillow, frame %d" % k
    assert durations == [pytest.approx(1000.0 * delay_num / delay_den)] * len(frames)
    assert A.strip_animation(apng) == P.encode(frames[0])
    assert len(apng) == A.size_identity([len(P.encode(f)) for f in frames], h)


def ref_payload(png, frame, n_frames, delay_num=1, delay_den=24):
    """Frame `frame`'s payload of an n_frames animation whose frame `frame` has the stand-alone PNG `png`."""
    return A.payloads_of_pngs([png] * n_frames, delay_num, delay_den)[frame]


NOISE = np.random.default_rng(4321).integers(0, 256, (37, 50, 3)).astype(np.uint8)


def noise_frames(h, n):
    rng = np.random.default_rng(h * 10 + n)
    return [rng.integers(0, 256, (h, 23, 3)).astype(np.uint8) for _ in range(n)]


def one_colour_frames(h, n):
    return [np.full((h, 41, 3), 30 + 40 * k, np.uint8) for k in range(n)]


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("h", [1, 15, 16, 17])
@pytest.mark.parametrize("kind", ["noise", "one_colour"])
def test_reference_writer(kind, h, n):
    frames = (noise_frames if kind == "noise" else one_colour_frames)(h, n)
    apng = A.encode(frames, 1, 24)
    check_animation(apng, frames, 1, 24)
    # each frame's payload stays within the per-frame bound
    for p in A.payloads(frames):
        assert len(p) <= A.frame_bound(P.bound(frames[0].shape[1], h), h)


def test_reference_writer_other_delay_and_sequence_numbers():
    frames = [NOISE, NOISE[::-1].copy(), np.full_like(NOISE, 9)]
    apng = A.encode(frames, 1, 7)
    check_animation(apng, frames, 1, 7)
    # s_f = 1 + (f - 1)(C + 1): C = 5 chunks of zlib data for 37 rows; the last number is (n - 1)(C + 1)
    _, _, fctls = A.walk(apng)
    assert [fc[0] for fc in fctls] == [0, 1, 7]
    assert A.fctl_seq(2, 37) + A.chunk_count(37) == (3 - 1) * (A.chunk_count(37) + 1)


def test_apng_bound_needs_no_device(rt):
    for (w, h) in [(1, 1), (17, 33), (1024, 768), (3840, 2160), (65535, 1), (1, 65535)]:
        for n in (1, 2, 120):
            assert rt.apng_bound(w, h, n) == A.frame_bound(P.bound(w, h), h)
    for (w, h, n) in [(0, 1, 1), (1, 0, 1), (65536, 1, 1), (1, 65536, 1), (5, 5, 0)]:
        with pytest.raises(rt.RtError) as e:
            rt.apng_bound(w, h, n)
        assert e.value.code == rt.RT_ERR_INVALID
    # the last sequence number (n - 1)(C + 1) must fit in 31 bits
    h = 65535
    n_max = (2 ** 31 - 1) // (A.chunk_count(h) + 1) + 1
    assert rt.apng_bound(1, h, n_max) > 0
    with pytest.raises(rt.RtError) as e:
        rt.apng_bound(1, h, n_max + 1)
    assert e.value.code == rt.RT_ERR_INVALID


# ---- command line without a device ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rtrace():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-s", "-C", ROOT, "rtrace"])
    return BIN


def run(rtrace, *args, cwd=None):
    return subprocess.run([rtrace] + list(args), capture_output=True, cwd=cwd, timeout=600)


def test_cli_apng_needs_the_png_extension(rtrace, tmp_path):
    r = run(rtrace, "--format", "apng", "--frames=3", "movie.tga", cwd=str(tmp_path))
    assert r.returncode == 0
    assert r.stdout == b"Output file 'movie.tga' must have the png extension, e.g. movie.png\n"
    assert not list(tmp_path.iterdir())


def test_cli_apng_usage_errors_and_help(rtrace, tmp_path):
    r = run(rtrace, "--format=apng", "--buckets", "o.png", cwd=str(tmp_path))
    assert r.returncode == 1 and b"--buckets" in r.stderr
    for args in (["--fps=12", "o.tga"], ["--fps", "12", "--format=png", "o.png"], ["--format=apng", "--fps=0", "o.png"],
                 ["--format=apng", "--fps=65536", "o.png"]):
        r = run(rtrace, *args, cwd=str(tmp_path))
        assert r.returncode == 1 and b"--fps" in r.stderr, args
    assert not list(tmp_path.iterdir())
    help_text = run(rtrace, "--help").stdout
    assert b"apng" in help_text and b"--fps <F>" in help_text


# ---- on the GPU -------------------------------------------------------------------------------------------------
class DeviceFrame:
    """A frame rendered into device memory, and its bytes on the host."""

    def __init__(self, rt, scene, w, h, spp, camera=None):
        self.rt, self.w, self.h = rt, w, h
        self.ptr = rt.device_alloc(w * h * 4)
        rt.Renderer.render(rt.RenderOptions(w, h, spp), scene, camera=camera, out_ptr=self.ptr)
        self.rgba = np.empty((h, w, 4), np.uint8)
        rt.memcpy(self.rgba.ctypes.data, self.ptr, self.rgba.nbytes)
        self.rgb = np.ascontiguousarray(self.rgba[:, :, :3])

    def close(self):
        self.rt.device_free(self.ptr)


POSITIONS = [(0, 1), (0, 3), (1, 3), (2, 3), (4, 7)]  # (frame, n_frames): first, middle, last, only


def check_payloads(rt, ptr, w, h, png, pitch=0):
    """Every position's payload of the device frame at `ptr` is the reference writer's for the PNG `png`."""
    for f, n in POSITIONS:
        got = rt.encode_apng_frame(ptr, w, h, f, n, fps=30, pitch=pitch)
        assert got == ref_payload(png, f, n, 1, 30), "frame %d of %d" % (f, n)
        assert len(got) <= rt.apng_bound(w, h, n)


@pytest.mark.gpu
def test_encode_apng_frame_on_c1(rt, gpu_scene8):
    f = DeviceFrame(rt, gpu_scene8, GOLD["width"], GOLD["height"], GOLD["spp"])
    try:
        png = P.encode(f.rgb)
        assert len(png) == 562214
        check_payloads(rt, f.ptr, f.w, f.h, png)
        one = rt.encode_apng_frame(f.ptr, f.w, f.h, 0, 1)
        assert A.strip_animation(one) == png
        assert hashlib.sha256(A.decode_frames(one)[0].tobytes()).hexdigest() == GOLD["rgb_sha256"]
    finally:
        f.close()


@pytest.mark.gpu
def test_encode_apng_frame_on_c5_orbit_frames(rt):
    """C5 orbit frames 7, 41 and 88 as frames of the 120-frame animation: the payload is the reference writer's
    (from the frame's PNG file, checked against the reference encoder in test_png) and decodes to rgb_sha256."""
    cases = DERIVED["c5_cases"]
    scene = rt.Scene(level=cases[0]["level"])
    for c in cases:
        f = DeviceFrame(rt, scene, c["width"], c["height"], c["spp"], camera=rt.orbit_camera(c["frame"], c["n_frames"]))
        try:
            assert hashlib.sha256(f.rgba.tobytes()).hexdigest() == c["rgba_sha256"], "orbit frame %d" % c["frame"]
            png = rt.encode_png(f.ptr, f.w, f.h)
            got = rt.encode_apng_frame(f.ptr, f.w, f.h, c["frame"], c["n_frames"])
            assert got == A.payloads_of_pngs([png] * c["n_frames"])[c["frame"]]
            ihdr = P.chunk(b"IHDR", P.chunks(png)[0][1])
            datas = [d[4:] for t, d in P.chunks(P.SIGNATURE + got) if t == b"fdAT"]
            dec = P.decode(P.SIGNATURE + ihdr + b"".join(P.chunk(b"IDAT", d) for d in datas) + P.chunk(b"IEND", b""))
            assert hashlib.sha256(dec.tobytes()).hexdigest() == c["rgb_sha256"], "orbit frame %d" % c["frame"]
        finally:
            f.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (17, 33), (65535, 1), (40, 15), (40, 16), (40, 17)])
def test_encode_apng_frame_odd_sizes(rt, gpu_scene8, w, h):
    f = DeviceFrame(rt, gpu_scene8, w, h, 2)
    try:
        check_payloads(rt, f.ptr, w, h, P.encode(f.rgb))
    finally:
        f.close()


@pytest.mark.gpu
def test_encode_apng_frame_pitched_and_synthetic(rt, gpu_scene8):
    w, h, spp = 203, 45, 2
    pitch = (w + 13) * 4
    ptr = rt.device_alloc(pitch * h)
    try:
        rt.Renderer.render_rows(rt.RenderOptions(w, h, spp), gpu_scene8, out_ptr=ptr, pitch=pitch, row_count=h)
        padded = np.empty((h, pitch), np.uint8)
        rt.memcpy(padded.ctypes.data, ptr, padded.nbytes)
        rgb = np.ascontiguousarray(padded[:, :w * 4].reshape(h, w, 4)[:, :, :3])
        check_payloads(rt, ptr, w, h, P.encode(rgb), pitch=pitch)
    finally:
        rt.device_free(ptr)
    rng = np.random.default_rng(11)
    runs = np.repeat(rng.integers(0, 256, (50, 4)), rng.integers(1, 400, 50), axis=0)[None].astype(np.uint8)
    frames = [rng.integers(0, 256, (33, 77, 4)).astype(np.uint8), np.full((33, 77, 4), 160, np.uint8)]
    for rgba in frames + [runs]:
        rgba = np.ascontiguousarray(rgba)
        hh, ww, _ = rgba.shape
        ptr = rt.device_alloc(rgba.nbytes)
        try:
            rt.memcpy(ptr, rgba.ctypes.data, rgba.nbytes)
            check_payloads(rt, ptr, ww, hh, P.encode(rgba[:, :, :3]))
        finally:
            rt.device_free(ptr)
    # two different frames make one animation that Pillow plays back
    ptrs = [rt.device_alloc(fr.nbytes) for fr in frames]
    try:
        for p, fr in zip(ptrs, frames):
            rt.memcpy(p, np.ascontiguousarray(fr).ctypes.data, fr.nbytes)
        apng = b"".join(rt.encode_apng_frame(p, 77, 33, k, 2) for k, p in enumerate(ptrs))
        check_animation(apng, [np.ascontiguousarray(fr[:, :, :3]) for fr in frames])
    finally:
        for p in ptrs:
            rt.device_free(p)


@pytest.mark.gpu
def test_encode_apng_frame_errors(rt, gpu_scene8):
    L = rt.lib()
    f = DeviceFrame(rt, gpu_scene8, 64, 48, 1)
    try:
        full = rt.encode_apng_frame(f.ptr, 64, 48, 1, 3)
        n = C.c_size_t()
        short = C.create_string_buffer(len(full) - 1)
        rc = L.rt_encode_apng_frame(C.c_void_p(f.ptr), 64, 48, 0, 1, 3, 1, 24, short, len(full) - 1, C.byref(n), None)
        assert rc == rt.RT_ERR_BUFFER and n.value == len(full)
        out = C.create_string_buffer(len(full))
        for frame, n_frames in [(3, 3), (0, 0), (7, 2)]:
            rc = L.rt_encode_apng_frame(C.c_void_p(f.ptr), 64, 48, 0, frame, n_frames, 1, 24, out, len(full), C.byref(n), None)
            assert rc == rt.RT_ERR_INVALID, (frame, n_frames)
        host = np.zeros((48, 64, 4), np.uint8)
        rc = L.rt_encode_apng_frame(C.c_void_p(host.ctypes.data), 64, 48, 0, 0, 1, 1, 24, out, len(full), C.byref(n), None)
        assert rc == rt.RT_ERR_INVALID
        assert L.rt_encode_apng_frame(C.c_void_p(f.ptr), 64, 48, 0, 1, 3, 1, 24, out, len(full), C.byref(n), None) == rt.RT_OK
        assert out.raw[:n.value] == full
    finally:
        f.close()


def apng_sweep(rt, scenes, w, h, spp, n, fps):
    cams = [rt.orbit_camera(k, 24) for k in range(n)]
    order, parts = [], []
    st = rt.Renderer.render_sweep_apng(rt.RenderOptions(w, h, spp), scenes, n, cameras=cams, fps=fps,
                                       on_frame=lambda k, b: (order.append(k), parts.append(b)))
    assert order == list(range(n)) and st.gpus == len(scenes)
    return cams, parts


@pytest.mark.gpu
def test_sweep_apng_single_gpu(rt, gpu_scene8):
    w, h, spp, n = 320, 200, 2, 7
    cams, parts = apng_sweep(rt, [gpu_scene8], w, h, spp, n, 12)
    rgbs = {}
    rt.Renderer.render_sweep_multi(rt.RenderOptions(w, h, spp), [gpu_scene8], n, cameras=cams, rgb=True,
                                   on_frame=lambda k, a: rgbs.__setitem__(k, a.copy()))
    frames = [rgbs[k] for k in range(n)]
    assert parts == A.payloads(frames, 1, 12)
    check_animation(b"".join(parts), frames, 1, 12)


@pytest.mark.gpu
def test_sweep_apng_two_gpus(rt, gpu_scene8):
    if rt.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    scenes = []
    for g in range(2):
        rt.set_device(g)
        scenes.append(rt.Scene())
    rt.set_device(0)
    _, one = apng_sweep(rt, [gpu_scene8], 320, 200, 2, 7, 24)
    _, two = apng_sweep(rt, scenes, 320, 200, 2, 7, 24)
    assert b"".join(two) == b"".join(one)


@pytest.mark.gpu
def test_sweep_apng_rejects_bad_animations(rt, gpu_scene8):
    with pytest.raises(rt.RtError) as e:
        rt.Renderer.render_sweep_apng(rt.RenderOptions(32, 32, 1), [gpu_scene8], 0)
    assert e.value.code == rt.RT_ERR_INVALID


@pytest.mark.gpu
def test_cli_apng_frames_are_one_file(rtrace, tmp_path):
    w, h = 160, 96
    a = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "a.tga", cwd=str(tmp_path))
    b = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "--format=apng", "--fps=10", "b.png",
            cwd=str(tmp_path))
    assert a.returncode == 0 and b.returncode == 0, b.stderr
    assert sorted(p.name for p in tmp_path.iterdir() if p.name.startswith("b")) == ["b.png"]
    hdr = len(b"P6\n160 96\n255\n")
    bodies = [np.frombuffer((tmp_path / ("a.%04d.tga" % k)).read_bytes()[hdr:], np.uint8).reshape(h, w, 3)
              for k in range(3)]
    apng = (tmp_path / "b.png").read_bytes()
    check_animation(apng, bodies, 1, 10)
    s = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--frames=3", "--format=apng", "--fps=10", "-")
    assert s.returncode == 0 and s.stdout == apng


@pytest.mark.gpu
def test_cli_apng_one_frame_is_the_png_file(rtrace, tmp_path):
    r = run(rtrace, "--format=apng", "--samples-per-pixel=4", "--width=1024", "--height=768", "out.png",
            cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr
    apng = (tmp_path / "out.png").read_bytes()
    png = A.strip_animation(apng)
    assert len(png) == 562214
    assert hashlib.sha256(P.decode(png).tobytes()).hexdigest() == GOLD["rgb_sha256"]
    _, actl, _ = A.walk(apng)
    assert actl == (1, 0)


@pytest.mark.gpu
def test_cli_apng_preview_frames(rtrace, tmp_path):
    w, h = 160, 96
    p = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--preview=4", "--frames=3", "--format=apng", "p.png",
            cwd=str(tmp_path))
    q = run(rtrace, "--width=%d" % w, "--height=%d" % h, "--preview=4", "--frames=3", "q.tga", cwd=str(tmp_path))
    assert p.returncode == 0 and q.returncode == 0, p.stderr
    assert sorted(x.name for x in tmp_path.iterdir() if x.name.startswith("p")) == ["p.png"]
    hdr = len(b"P6\n160 96\n255\n")
    bodies = [np.frombuffer((tmp_path / ("q.%04d.tga" % k)).read_bytes()[hdr:], np.uint8).reshape(h, w, 3)
              for k in range(3)]
    check_animation((tmp_path / "p.png").read_bytes(), bodies)
