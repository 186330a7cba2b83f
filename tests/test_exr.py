"""OpenEXR output encoded on the GPU: rt_encode_exr, rt_exr_bound and `rtrace --format exr [--aov]`.

The layout is fixed (include/rtrace.h "OpenEXR output", tests/_exr_ref.py), so the GPU's file is compared with the
reference encoder's byte for byte.  The CPU part ties the reference encoder to the float and AOV oracles (its files
decode, through its own decoder and through OpenEXR in OpenCV, to the oracle's floats bit for bit), checks its parse
against a byte-by-byte restatement of the rule, and checks the command line; the GPU part checks the encoder and the
CLI against the reference."""
import os

os.environ["OPENCV_IO_ENABLE_OPENEXR"] = "1"   # before OpenCV is imported anywhere

import subprocess
import sys
import zlib

import numpy as np
import pytest

import _exr_ref as X
import _oracle_aov
import _oracle_f32

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "target", "release", "rtrace")


def run(cmd, *args, cwd=None, timeout=600):
    return subprocess.run([cmd] + list(args), capture_output=True, cwd=cwd, timeout=timeout)


@pytest.fixture(scope="module")
def rtrace():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-s", "-C", ROOT, "rtrace"])
    return BIN


def cv2_exr():
    try:
        import cv2
    except ImportError:
        return None
    return cv2


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a, np.float32).view(np.uint32),
                                                 np.ascontiguousarray(b, np.float32).view(np.uint32))


def check_file(data, rgba, aov, tmp_path=None):
    """`data` decodes (reference decoder, and OpenEXR through OpenCV when it has EXR) to the frames bit for bit."""
    dec = X.decode(data)
    assert list(dec) == X.NAMES[:4 if aov is None else 12]
    for name, plane in zip(X.NAMES, X.channel_planes(rgba, aov)):
        assert bits_equal(dec[name], plane), name
    cv2 = cv2_exr()
    if cv2 is not None and tmp_path is not None:
        p = str(tmp_path / "check.exr")
        with open(p, "wb") as f:
            f.write(data)
        try:
            img = cv2.imread(p, cv2.IMREAD_UNCHANGED)
        except cv2.error:
            img = None
        if img is not None:   # OpenCV reads the RGBA layer as B, G, R, A
            h, w = rgba.shape[:2]
            assert bits_equal(img.reshape(h, w, 4), rgba[..., [2, 1, 0, 3]])


# ---- CPU ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,spp", [(1, 1, 1), (37, 21, 2), (64, 48, 3), (100, 17, 4), (24, 16, 5), (20, 31, 6),
                                     (17, 9, 7), (16, 8, 8), (12, 40, 9), (160, 90, 2)])
def test_reference_files_decode_to_the_oracle(w, h, spp, tmp_path):
    rgba = _oracle_f32.Scene().render_f32(w, h, spp)[0]
    aov = _oracle_aov.Scene().render_aov(w, h, spp)
    for a in (None, aov):
        data = X.encode(rgba, a)
        check_file(data, rgba, a, tmp_path)
        assert len(data) <= X.bound(w, h, a is not None)


@pytest.mark.parametrize("frame", [0, 7, 41])
def test_reference_files_orbit_cameras(oracle, frame, tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    cam = oracle.make_camera(*bench.orbit_basis(frame))
    w, h, spp = 120, 90, 2
    rgba = _oracle_f32.Scene().render_f32(w, h, spp, camera=cam)[0]
    aov = _oracle_aov.Scene().render_aov(w, h, spp, camera=cam)
    check_file(X.encode(rgba, aov), rgba, aov, tmp_path)


def test_reference_without_d2(tmp_path):
    """W > 16384: 2W is beyond deflate's window, so there is no far distance."""
    w, h = 16385, 3
    rgba = _oracle_f32.Scene().render_f32(w, h, 1)[0]
    aov = _oracle_aov.Scene().render_aov(w, h, 1)
    data = X.encode(rgba, aov)
    check_file(data, rgba, aov)
    assert X.chunk_kinds(data) == [False]


def test_parse_rule_matches_the_byte_by_byte_statement():
    rgba = _oracle_f32.Scene().render_f32(37, 21, 2)[0]
    aov = _oracle_aov.Scene().render_aov(37, 21, 2)
    planes = X.channel_planes(rgba, aov)
    cases = [(X.predict(X.chunk_raw(planes, 0, 16)), 74), (X.predict(X.chunk_raw(planes[:4], 16, 21)), 74)]
    rng = np.random.default_rng(5)
    runs = np.repeat(rng.integers(0, 4, 700), rng.integers(1, 90, 700)).astype(np.uint8)[:40000]
    cases += [(runs, 6), (runs, 0), (np.full(20000, 7, np.uint8), 2), (rng.integers(0, 256, 300).astype(np.uint8), 8)]
    for d, d2 in cases:
        z = X.zlib_stream(d, d2)
        assert z == X.slow_stream(d, d2)
        assert zlib.decompress(z) == d.tobytes()


def test_random_floats_fall_back_to_raw_chunks(tmp_path):
    rng = np.random.default_rng(3)
    rgba = rng.standard_normal((40, 30, 4)).astype(np.float32)
    aov = rng.standard_normal((40, 30, 8)).astype(np.float32)
    for a in (None, aov):
        data = X.encode(rgba, a)
        assert X.chunk_kinds(data) == [True] * 3 and len(data) == X.bound(30, 40, a is not None)
        check_file(data, rgba, a, tmp_path)


def test_bound_arithmetic(rt):
    for w, h in ((1, 1), (37, 21), (1024, 768), (16385, 3), (65535, 65535)):
        for aov in (False, True):
            assert rt.exr_bound(w, h, aov) == X.bound(w, h, aov)
    n = rt.C.c_size_t()
    for w, h in ((0, 5), (5, 0), (65536, 1), (1, 65536)):
        assert rt.lib().rt_exr_bound(w, h, 0, rt.C.byref(n)) == rt.RT_ERR_INVALID


def test_cli_exr_arguments(rtrace, tmp_path):
    for args, flag in ((["--format=exr", "--buckets", "o.exr"], b"--buckets"),
                       (["--format=exr", "--preview=4", "o.exr"], b"--preview"),
                       (["--format=exr", "--aov", "--buckets", "o.exr"], b"--buckets"),
                       (["--format=png", "--aov", "o.png"], b"'--format exr'"),
                       (["--format=exf", "o.tga"], b"exr")):
        r = run(rtrace, *args, cwd=str(tmp_path))
        assert r.returncode == 1 and flag in r.stderr, (args, r.stderr)
    r = run(rtrace, "--format=exr", "--aov", "picture.pfm", cwd=str(tmp_path))
    assert r.returncode == 0 and b"must have the exr extension" in r.stdout
    assert not list(tmp_path.iterdir())
    h = run(rtrace, "--help").stdout
    assert b"--format exr" in h and b".exr" in h


# ---- GPU ----------------------------------------------------------------------------------------------------------
def gpu_frames(rt, scene, w, h, spp, camera=None):
    import torch
    rgba = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    aov = torch.empty((h, w, 8), dtype=torch.float32, device="cuda")
    rt.Renderer.render_f32(rt.RenderOptions(w, h, spp), scene, camera=camera, out_ptr=rgba.data_ptr())
    rt.Renderer.render_aov(rt.RenderOptions(w, h, spp), scene, camera=camera, out_ptr=aov.data_ptr())
    return rgba, aov


def encode_both(rt, rgba, aov):
    h, w = rgba.shape[:2]
    return rt.encode_exr(rgba.data_ptr(), w, h), rt.encode_exr(rgba.data_ptr(), w, h, aov_ptr=aov.data_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,spp,level", [(1024, 768, 4, 8), (3840, 2160, 1, 8), (3840, 2160, 4, 9),
                                          (7680, 4320, 4, 9)], ids=["C1", "C2", "C3", "C4"])
def test_encode_exr_baseline_frames(rt, w, h, spp, level):
    scene = rt.Scene(level=level)
    rgba, aov = gpu_frames(rt, scene, w, h, spp)
    scene.close()
    colour, full = encode_both(rt, rgba, aov)
    r, a = rgba.cpu().numpy(), aov.cpu().numpy()
    assert colour == X.encode(r)
    if w * h <= 3840 * 2160:   # the reference's 12-channel C4 file would take minutes on the CPU
        assert full == X.encode(r, a)
    else:
        check_file(full, r, a)
    assert not any(X.chunk_kinds(colour))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,spp", [(1, 1, 1), (37, 21, 2), (100, 17, 3), (333, 50, 5), (64, 48, 9), (16385, 3, 1),
                                     (16384, 2, 1), (20000, 40, 1)])
def test_encode_exr_odd_sizes_and_no_d2(rt, gpu_scene8, w, h, spp, tmp_path):
    rgba, aov = gpu_frames(rt, gpu_scene8, w, h, spp)
    colour, full = encode_both(rt, rgba, aov)
    r, a = rgba.cpu().numpy(), aov.cpu().numpy()
    assert colour == X.encode(r)
    assert full == X.encode(r, a)
    check_file(full, r, a, tmp_path)


@pytest.mark.gpu
def test_encode_exr_orbit_frames(rt, gpu_scene8):
    for f in (3, 17):
        rgba, aov = gpu_frames(rt, gpu_scene8, 320, 180, 2, camera=rt.orbit_camera(f, 48))
        assert encode_both(rt, rgba, aov) == (X.encode(rgba.cpu().numpy()),
                                              X.encode(rgba.cpu().numpy(), aov.cpu().numpy()))


@pytest.mark.gpu
def test_encode_exr_random_floats_are_stored_raw(rt):
    import torch
    g = torch.Generator(device="cuda").manual_seed(11)
    for w, h in ((1000, 70), (31, 5)):
        rgba = torch.randn((h, w, 4), device="cuda", generator=g)
        aov = torch.randn((h, w, 8), device="cuda", generator=g)
        colour, full = encode_both(rt, rgba, aov)
        r, a = rgba.cpu().numpy(), aov.cpu().numpy()
        assert colour == X.encode(r) and full == X.encode(r, a)
        assert all(X.chunk_kinds(colour)) and all(X.chunk_kinds(full))
        assert len(full) == rt.exr_bound(w, h, True)


@pytest.mark.gpu
def test_encode_exr_pitched_inputs_and_device_output(rt, gpu_scene8):
    import torch
    w, h, spp = 200, 70, 2
    rgba, aov = gpu_frames(rt, gpu_scene8, w, h, spp)
    want = X.encode(rgba.cpu().numpy(), aov.cpu().numpy())
    prgba = torch.full((h, w * 4 + 8), -3.0, device="cuda")
    paov = torch.full((h, w * 8 + 4), -5.0, device="cuda")
    prgba[:, :w * 4] = rgba.reshape(h, w * 4)
    paov[:, :w * 8] = aov.reshape(h, w * 8)
    got = rt.encode_exr(prgba.data_ptr(), w, h, aov_ptr=paov.data_ptr(), pitch=(w * 4 + 8) * 4, aov_pitch=(w * 8 + 4) * 4)
    assert got == want
    L, n = rt.lib(), rt.C.c_size_t()
    cap = rt.exr_bound(w, h, True)
    dout = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        assert L.rt_encode_exr(rgba.data_ptr(), 0, aov.data_ptr(), 0, w, h, dout.data_ptr(), cap, rt.C.byref(n),
                               torch.cuda.current_stream().cuda_stream) == rt.RT_OK
    assert n.value == len(want) and bytes(dout[:n.value].cpu().numpy()) == want


@pytest.mark.gpu
def test_encode_exr_error_codes(rt, gpu_scene8):
    import torch
    L, n, w, h = rt.lib(), rt.C.c_size_t(), 64, 32
    rgba, aov = gpu_frames(rt, gpu_scene8, w, h, 1)
    want = X.encode(rgba.cpu().numpy(), aov.cpu().numpy())
    out = rt.C.create_string_buffer(rt.exr_bound(w, h, True))
    cap = len(out)

    def enc(r=rgba.data_ptr(), rp=0, a=aov.data_ptr(), ap=0, ww=w, hh=h, o=out, c=cap):
        return L.rt_encode_exr(r, rp, a, ap, ww, hh, o, c, rt.C.byref(n), None)

    host = np.zeros((h, w, 8), np.float32)
    assert enc(r=host.ctypes.data) == rt.RT_ERR_INVALID          # host frames
    assert enc(a=host.ctypes.data) == rt.RT_ERR_INVALID
    assert enc(r=rgba.data_ptr() + 4) == rt.RT_ERR_INVALID       # misaligned
    assert enc(a=aov.data_ptr() + 8) == rt.RT_ERR_INVALID
    assert enc(rp=w * 16 + 4) == rt.RT_ERR_INVALID               # pitch not a multiple of 16
    assert enc(rp=w * 16 - 16) == rt.RT_ERR_INVALID              # pitch shorter than a row
    assert enc(ap=w * 32 - 16) == rt.RT_ERR_INVALID
    assert enc(ww=0) == rt.RT_ERR_INVALID and enc(hh=0) == rt.RT_ERR_INVALID
    assert enc(r=None) == rt.RT_ERR_INVALID
    assert enc(c=len(want) - 1) == rt.RT_ERR_BUFFER and n.value == len(want)
    assert enc(o=None, c=0) == rt.RT_ERR_BUFFER and n.value == len(want)
    assert enc(c=len(want)) == rt.RT_OK and out.raw[:n.value] == want
    torch.cuda.synchronize()


def cli_expected(oracle, w, h, spp, aov, frames=1):
    sys.path.insert(0, ROOT)
    import bench
    files = []
    for f in range(frames):
        cam = oracle.make_camera(*bench.orbit_basis(f, frames)) if frames > 1 else None
        rgba = _oracle_f32.Scene().render_f32(w, h, spp, camera=cam)[0]
        files.append(X.encode(rgba, _oracle_aov.Scene().render_aov(w, h, spp, camera=cam) if aov else None))
    return files


@pytest.mark.gpu
def test_cli_exr_matches_reference(rtrace, oracle, tmp_path):
    w, h, spp = 1024, 768, 4
    args = ["--format=exr", "--width=%d" % w, "--height=%d" % h, "--samples-per-pixel=%d" % spp]
    colour, full = cli_expected(oracle, w, h, spp, False)[0], cli_expected(oracle, w, h, spp, True)[0]
    r = run(rtrace, *args, "out.exr", cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout == b"", r.stderr
    assert (tmp_path / "out.exr").read_bytes() == colour
    r = run(rtrace, *args, "--aov", "--stats", "full.exr", cwd=str(tmp_path))
    assert r.returncode == 0 and b"kernel" in r.stderr, r.stderr
    assert (tmp_path / "full.exr").read_bytes() == full
    r = run(rtrace, *args, "--aov", "-", cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout == full
    assert sorted(p.name for p in tmp_path.iterdir()) == ["full.exr", "out.exr"]


@pytest.mark.gpu
def test_cli_exr_frames_and_gpus(rt, rtrace, oracle, tmp_path):
    w, h, spp, n = 160, 90, 2, 3
    want = cli_expected(oracle, w, h, spp, True, n)
    for gpus in sorted({1, min(2, rt.device_count())}):
        d = tmp_path / ("g%d" % gpus)
        d.mkdir()
        r = run(rtrace, "--format=exr", "--aov", "--frames=%d" % n, "--gpus=%d" % gpus, "--width=%d" % w,
                "--height=%d" % h, "--samples-per-pixel=%d" % spp, "s.exr", cwd=str(d))
        assert r.returncode == 0, r.stderr
        assert sorted(p.name for p in d.iterdir()) == ["s.%04d.exr" % f for f in range(n)]
        for f in range(n):
            assert (d / ("s.%04d.exr" % f)).read_bytes() == want[f], (gpus, f)
        r = run(rtrace, "--format=exr", "--frames=%d" % n, "--gpus=%d" % gpus, "--width=%d" % w, "--height=%d" % h,
                "--samples-per-pixel=%d" % spp, "-", cwd=str(d))
        assert r.returncode == 0 and r.stdout == b"".join(cli_expected(oracle, w, h, spp, False, n))


@pytest.mark.gpu
def test_cli_exr_two_gpus(rt, rtrace, oracle, tmp_path):
    if rt.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    w, h, spp = 640, 480, 2
    r = run(rtrace, "--format=exr", "--aov", "--gpus=2", "--width=%d" % w, "--height=%d" % h,
            "--samples-per-pixel=%d" % spp, "o.exr", cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "o.exr").read_bytes() == cli_expected(oracle, w, h, spp, True)[0]
