"""Float output: rt_render_rows_f32, rt_render_frame_multi_f32 and `rtrace --format pfm`.

A float frame holds each pixel before quantisation, {r, g, b, alpha} times 1/(spp*spp) (render.rs:249-250), and must
equal the oracle's f32 values bit for bit.  Quantised with the reference's rule (render.rs:96-103) it is the RGBA8
frame.  The CPU part checks that identity on the oracle itself, the PFM writer and the CLI's argument handling; the
GPU part checks the kernels (PHASED and its LANE fallback) against the oracle."""
import hashlib
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import _oracle_f32

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "target", "release", "rtrace")
SELFTEST = os.path.join(ROOT, "target", "release", "rtrace_selftest")
GOLD = json.load(open(os.path.join(HERE, "golden", "rtrace_output_1024x768.json")))
F32_GOLD = json.load(open(os.path.join(HERE, "golden", "oracle_f32.json")))


def quantise(v):
    """render.rs:96-103: trunc(0.5 + 255 v) in f32, > 255 -> 255, NaN or <= 0 -> 0."""
    r = np.float32(0.5) + np.float32(255.0) * np.asarray(v, np.float32)
    with np.errstate(invalid="ignore"):
        r = np.where(r > np.float32(255.0), np.float32(255.0), np.where(r > np.float32(0.0), r, np.float32(0.0)))
    return np.trunc(r).astype(np.uint8)


def assert_bits(got, ref, what=""):
    """Equal bit for bit (a float compare would let -0.0 == 0.0 and NaN != NaN pass or fail wrongly)."""
    assert got.shape == ref.shape and got.dtype == np.float32, (what, got.shape, got.dtype)
    g, r = got.view(np.uint32), ref.view(np.uint32)
    if not np.array_equal(g, r):
        ys, xs = np.nonzero((g != r).any(axis=-1))
        raise AssertionError("%s: %d of %d pixels differ, first at row %d col %d: gpu %r ref %r" % (
            what, len(ys), g.shape[0] * g.shape[1], ys[0], xs[0], got[ys[0], xs[0]], ref[ys[0], xs[0]]))


def f32_sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<f4").tobytes()).hexdigest()


@pytest.fixture(scope="module")
def rtrace():
    if not (os.path.exists(BIN) and os.path.exists(SELFTEST)):
        subprocess.check_call(["make", "-s", "-C", ROOT, "rtrace"])
    return BIN


def run(cmd, *args, cwd=None, timeout=300):
    return subprocess.run([cmd] + list(args), capture_output=True, cwd=cwd, timeout=timeout)


@pytest.fixture(scope="module")
def f32_scene8():
    """The default scene (level 8) in the float oracle."""
    return _oracle_f32.Scene()


def pfm_bytes(rgba):
    """What `rtrace --format pfm` writes for a float frame: header, then RGB rows bottom-up, little-endian."""
    h, w, _ = rgba.shape
    return b"PF\n%d %d\n-1.0\n" % (w, h) + np.ascontiguousarray(rgba[::-1, :, :3], dtype="<f4").tobytes()


# ---- CPU: the oracle's float values, the PFM writer, the command line ---------------------------------------------
@pytest.mark.parametrize("w,h,spp,level", [(64, 48, 1, 2), (33, 7, 2, 8), (40, 30, 3, 5), (97, 61, 4, 9),
                                          (24, 16, 5, 3), (20, 12, 6, 8), (17, 9, 7, 6), (16, 8, 8, 8),
                                          (12, 8, 9, 4), (1, 1, 1, 8), (32, 18, 1, 10), (24, 12, 2, 11),
                                          (16, 9, 1, 12)])
def test_quantised_oracle_f32_is_the_rgba8_frame(oracle, w, h, spp, level):
    f, fc = _oracle_f32.Scene(level=level).render_f32(w, h, spp)
    b, bc = oracle.Scene(level=level).render(w, h, spp)   # the pinned oracle's own library
    assert np.array_equal(quantise(f), b)
    assert fc.as_dict() == bc.as_dict()   # the same rays were traced
    assert np.array_equal(f[..., 1].view(np.uint32), f[..., 2].view(np.uint32))   # blue == green (render.rs:172-186)


@pytest.mark.parametrize("frame", [0, 7, 41, 88])
def test_quantised_oracle_f32_orbit_and_rows(oracle, frame):
    sys.path.insert(0, ROOT)
    import bench
    s = _oracle_f32.Scene(level=8)
    cam = oracle.make_camera(*bench.orbit_basis(frame))
    f, _ = s.render_f32(120, 90, 2, camera=cam)
    b, _ = oracle.Scene(level=8).render(120, 90, 2, camera=cam)
    assert np.array_equal(quantise(f), b)
    rows, _ = s.render_f32(120, 90, 2, row_start=1, row_stride=3, camera=cam)
    assert_bits(rows, f[1::3], "rows 1, 4, 7, ...")


def test_c1_quantised_equals_the_reference_image(f32_scene8):
    """C1 (`make image`) as floats, quantised: the reference's shipped image, row for row."""
    f, _ = f32_scene8.render_f32(GOLD["width"], GOLD["height"], GOLD["spp"])
    rgb = np.ascontiguousarray(quantise(f)[:, :, :3])
    bad = [y for y in range(GOLD["height"]) if zlib.crc32(rgb[y].tobytes()) != GOLD["row_crc32"][y]]
    assert not bad, bad[:10]
    c1 = [c for c in F32_GOLD["cases"] if (c["width"], c["height"], c["spp"], c["level"]) == (1024, 768, 4, 8)]
    assert len(c1) == 1 and f32_sha(f) == c1[0]["f32_sha256"]


def test_pfm_writer_layout(rtrace, tmp_path):
    """write_pfm (host/render.hpp) on the selftest's synthetic 3x2 frame: header, little-endian f32 RGB, bottom row
    first, alpha dropped, the source pitch followed."""
    r = run(SELFTEST, "pfm", str(tmp_path / "t.pfm"))
    assert r.returncode == 0 and b"ok pfm" in r.stdout, r.stderr
    px = (np.arange(24, dtype=np.float32) / np.float32(7.0)).reshape(2, 3, 4)
    data = (tmp_path / "t.pfm").read_bytes()
    assert data == pfm_bytes(px)
    assert data.startswith(b"PF\n3 2\n-1.0\n") and len(data) == 12 + 2 * 3 * 12
    first = np.frombuffer(data[12:24], "<f4")
    assert np.array_equal(first, px[1, 0, :3])   # the file starts with the bottom row


def test_cli_pfm_arguments(rtrace, tmp_path):
    r = run(rtrace, "--format=pfm", "picture.tga", cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout == b"Output file 'picture.tga' must have the pfm extension, e.g. picture.pfm\n"
    r = run(rtrace, "--format", "pfm", "picture", cwd=str(tmp_path))
    assert r.returncode == 0 and b"must have the pfm extension" in r.stdout
    for args, flag in ((["--buckets"], b"--buckets"), (["--preview=4"], b"--preview"), (["--fps=12"], b"--fps")):
        r = run(rtrace, "--format=pfm", *args, "o.pfm", cwd=str(tmp_path))
        assert r.returncode == 1 and flag in r.stderr, args
    assert not list(tmp_path.iterdir())
    h = run(rtrace, "--help").stdout
    assert b"--format pfm" in h and b".pfm" in h


# ---- GPU ----------------------------------------------------------------------------------------------------------
def expected_variant(rt, scene, w, h, spp, variant, camera=None):
    """The f32 variant rule, from what RGBA8 runs: LANE for a forced LANE or WARP; for a forced TILE or PHASED what a
    forced PHASED runs (PHASED inside its domain, LANE outside); AUTO: PHASED where RGBA8 runs TILE or PHASED."""
    if variant in (rt.VARIANT_LANE, rt.VARIANT_WARP):
        return rt.VARIANT_LANE
    rt.set_variant(rt.VARIANT_PHASED if variant != rt.VARIANT_AUTO else rt.VARIANT_AUTO)
    try:
        _, st = rt.Renderer.render(rt.RenderOptions(w, h, spp), scene, camera=camera, want_stats=True)
    finally:
        rt.set_variant(rt.VARIANT_AUTO)
    return rt.VARIANT_LANE if st.variant_used == rt.VARIANT_LANE else rt.VARIANT_PHASED


ALL_VARIANTS = ("VARIANT_AUTO", "VARIANT_LANE", "VARIANT_WARP", "VARIANT_TILE", "VARIANT_PHASED")


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,spp,level", [(64, 128, 2, 8), (160, 120, 1, 8), (160, 120, 3, 8), (200, 150, 4, 5),
                                          (97, 61, 2, 9), (256, 144, 1, 10), (33, 7, 1, 8), (1, 1, 1, 8), (8, 4, 5, 2),
                                          (320, 180, 5, 7), (200, 120, 6, 8), (131, 77, 7, 6), (256, 144, 8, 8),
                                          (40, 30, 9, 5), (96, 54, 1, 11), (48, 27, 2, 12)])
def test_f32_frame_matches_oracle(rt, w, h, spp, level):
    gs, os_ = rt.Scene(level=level), _oracle_f32.Scene(level=level)
    ref, _ = os_.render_f32(w, h, spp)
    for name in ALL_VARIANTS:
        v = getattr(rt, name)
        want = expected_variant(rt, gs, w, h, spp, v)
        rt.set_variant(v)
        try:
            img, st = rt.Renderer.render_f32(rt.RenderOptions(w, h, spp), gs, want_stats=True)
        finally:
            rt.set_variant(rt.VARIANT_AUTO)
        assert_bits(img, ref, "%s %dx%d spp %d L%d" % (name, w, h, spp, level))
        assert st.variant_used == want, (name, st.variant_used, want)
        assert st.kernel_launches == (4 if want == rt.VARIANT_PHASED else 1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", F32_GOLD["cases"],
                         ids=lambda c: "%dx%d_spp%d_L%d" % (c["width"], c["height"], c["spp"], c["level"]))
def test_f32_baseline_frames_match_fixture(rt, case):
    """Every BASELINE configuration at full size (C1, C2 at levels 8/9/10, C3, C4) against the oracle's float hash,
    on PHASED (what AUTO runs there) and on the forced LANE fallback."""
    gs = rt.Scene(level=case["level"])
    o = rt.RenderOptions(case["width"], case["height"], case["spp"])
    img, st = rt.Renderer.render_f32(o, gs, want_stats=True)
    assert st.variant_used == rt.VARIANT_PHASED
    assert f32_sha(img) == case["f32_sha256"]
    assert hashlib.sha256(quantise(img).tobytes()).hexdigest() == case["rgba_sha256"]
    rt.set_variant(rt.VARIANT_LANE)
    try:
        img, st = rt.Renderer.render_f32(o, gs, want_stats=True)
    finally:
        rt.set_variant(rt.VARIANT_AUTO)
    assert st.variant_used == rt.VARIANT_LANE and f32_sha(img) == case["f32_sha256"]


@pytest.mark.gpu
def test_f32_c5_orbit_frames_match_fixture(rt):
    cases = F32_GOLD["c5_cases"]
    gs = rt.Scene(level=cases[0]["level"])
    for c in cases:
        o = rt.RenderOptions(c["width"], c["height"], c["spp"])
        img, st = rt.Renderer.render_f32(o, gs, camera=rt.orbit_camera(c["frame"], c["n_frames"]), want_stats=True)
        assert st.variant_used == rt.VARIANT_PHASED
        assert f32_sha(img) == c["f32_sha256"], "orbit frame %d" % c["frame"]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,spp,level", [(3840, 2160, 4, 9), (7680, 4320, 4, 9)])   # C3, C4
def test_quantised_f32_is_the_rgba8_frame(rt, w, h, spp, level):
    gs = rt.Scene(level=level)
    o = rt.RenderOptions(w, h, spp)
    assert np.array_equal(quantise(rt.Renderer.render_f32(o, gs)), rt.Renderer.render(o, gs))


def _fallback_cases(rt, oracle):
    light = np.array([-1.0, -3.0, 2.0], np.float32)
    light /= np.float32(np.sqrt(np.float32((light * light).sum())))
    sph = np.array([[0, -1, 0, 2], [-0.6, -1, 0, 0.5], [0.6, -1, 0.3, 0.5], [0, -0.2, 0, 0.4]], np.float32)
    skip = np.array([4, 2, 3, 4], np.uint32)
    yield ("level 11", lambda: (rt.Scene(level=11), _oracle_f32.Scene(level=11)), (96, 54, 1), None)
    yield ("hand-built group", lambda: (rt.Scene.from_nodes(sph, skip, light, (0, 0, -4)),
                                        _oracle_f32.Scene.from_nodes(sph, skip, light, (0, 0, -4))), (80, 60, 2), None)
    yield ("spp 9", lambda: (rt.Scene(), _oracle_f32.Scene()), (40, 30, 9), None)
    yield ("eye inside the root bound", lambda: (rt.Scene(eye=(0.0, -0.6, -0.3)), _oracle_f32.Scene(eye=(0.0, -0.6, -0.3))),
           (64, 48, 2), None)
    yield ("non-orthonormal basis", lambda: (rt.Scene(), _oracle_f32.Scene()), (96, 64, 2),
           ((0.0, 0.0, -4.0), (1.01, 0.0, 0.0), (0.0, 1.0, 0.0), (0.0, 0.0, 1.0)))


@pytest.mark.gpu
def test_f32_fallbacks_run_lane_and_match_oracle(rt, oracle):
    for what, make, (w, h, spp), cam in _fallback_cases(rt, oracle):
        gs, os_ = make()
        ref, _ = os_.render_f32(w, h, spp, camera=oracle.make_camera(*cam) if cam else None)
        for name in ("VARIANT_AUTO", "VARIANT_PHASED", "VARIANT_TILE"):
            rt.set_variant(getattr(rt, name))
            try:
                img, st = rt.Renderer.render_f32(rt.RenderOptions(w, h, spp), gs,
                                                 camera=rt.make_camera(*cam) if cam else None, want_stats=True)
            finally:
                rt.set_variant(rt.VARIANT_AUTO)
            assert st.variant_used == rt.VARIANT_LANE, (what, name)
            assert_bits(img, ref, "%s (%s)" % (what, name))
        gs.close()


@pytest.mark.gpu
def test_f32_rows_pitch_and_host_memory(rt, f32_scene8, gpu_scene8):
    """Strided rows, a pitch wider than the row, pageable and pinned host memory."""
    import torch
    w, h, spp = 200, 150, 2
    o = rt.RenderOptions(w, h, spp)
    full, _ = f32_scene8.render_f32(w, h, spp)
    for variant in (rt.VARIANT_AUTO, rt.VARIANT_PHASED, rt.VARIANT_LANE):
        rt.set_variant(variant)
        try:
            rows = rt.Renderer.render_rows_f32(o, gpu_scene8, row_start=2, row_stride=3)
            assert_bits(rows, full[2::3], "rows 2, 5, 8, ...")
            pitch = w * 16 + 48
            buf = np.full((h, pitch // 4), np.float32(-7.0), np.float32)   # pageable, padded rows
            rt.Renderer.render_rows_f32(o, gpu_scene8, out_ptr=buf.ctypes.data, pitch=pitch)
            assert_bits(np.ascontiguousarray(buf[:, :w * 4]).reshape(h, w, 4), full, "pitched host rows")
            assert (buf[:, w * 4:] == np.float32(-7.0)).all()   # the padding is left alone
            pinned = torch.empty((h, w, 4), dtype=torch.float32, pin_memory=True)
            rt.Renderer.render_rows_f32(o, gpu_scene8, out_ptr=pinned.data_ptr())
            assert_bits(pinned.numpy(), full, "pinned host frame")
        finally:
            rt.set_variant(rt.VARIANT_AUTO)


@pytest.mark.gpu
def test_f32_into_a_torch_cuda_tensor(rt, f32_scene8, gpu_scene8):
    """Device output on torch's current stream: asynchronous, ordered with torch's own work on that stream."""
    import torch
    w, h, spp = 320, 240, 4
    o = rt.RenderOptions(w, h, spp)
    ref, _ = f32_scene8.render_f32(w, h, spp)
    dev = torch.device("cuda", gpu_scene8.device())
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.device(dev), torch.cuda.stream(side):
        t = torch.full((h, w, 4), float("nan"), dtype=torch.float32, device=dev)
        rt.Renderer.render_rows_f32(o, gpu_scene8, out_ptr=t.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        total = t.sum(dim=(0, 1))   # queued behind the render on the same stream
        pitched = torch.full((h, w * 4 + 8), -1.0, dtype=torch.float32, device=dev)
        rt.Renderer.render_rows_f32(o, gpu_scene8, out_ptr=pitched.data_ptr(), pitch=(w * 4 + 8) * 4,
                                    stream=torch.cuda.current_stream().cuda_stream)
        got, got_pitched, total = t.cpu().numpy(), pitched.cpu().numpy(), total.cpu().numpy()
    assert_bits(got, ref, "torch tensor")
    assert_bits(np.ascontiguousarray(got_pitched[:, :w * 4]).reshape(h, w, 4), ref, "pitched torch tensor")
    assert (got_pitched[:, w * 4:] == -1.0).all()
    assert np.isfinite(total).all()
    dframe = torch.empty((h, w, 4), dtype=torch.float32, device=dev)
    assert rt.Renderer.render_f32(o, gpu_scene8, out_ptr=dframe.data_ptr()) is None
    assert_bits(dframe.cpu().numpy(), ref, "rt_render_frame_multi_f32, device output")


SHAPE_SCRIPT = r"""
import json, sys
import numpy as np
import rtrace_b200 as rt
cases = json.loads(sys.argv[1])
scene = rt.Scene()
used = {}
for i, (variant, w, h, spp) in enumerate(cases):
    rt.set_variant(variant)
    img, st = rt.Renderer.render_f32(rt.RenderOptions(w, h, spp), scene, want_stats=True)
    np.save("%s/%d.npy" % (sys.argv[2], i), img)
    used[i] = int(st.variant_used)
json.dump(used, open(sys.argv[2] + "/used.json", "w"))
scene.close()
"""


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [0, 1, 2, 3, 4, 5, 6])
def test_f32_every_tile_shape(rt, f32_scene8, shape, tmp_path):
    """RTRACE_TILE_SHAPE (read once per process, so each shape runs in a process of its own) forces every
    spp-1 tile shape of PHASED, and the 4x4 shape of spp 2 and 4 where it exists."""
    cases = [(rt.VARIANT_PHASED, 173, 91, 1), (rt.VARIANT_PHASED, 1920, 1080, 1), (rt.VARIANT_PHASED, 130, 70, 2),
             (rt.VARIANT_PHASED, 96, 64, 4), (rt.VARIANT_TILE, 61, 47, 1)]
    env = dict(os.environ, RTRACE_TILE_SHAPE=str(shape),
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "rust-tracer_b200"), HERE]))
    subprocess.run([sys.executable, "-c", SHAPE_SCRIPT, json.dumps(cases), str(tmp_path)], env=env, check=True,
                   timeout=900)
    used = json.loads((tmp_path / "used.json").read_text())
    for i, (variant, w, h, spp) in enumerate(cases):
        assert used[str(i)] == rt.VARIANT_PHASED, (i, used[str(i)])
        ref, _ = f32_scene8.render_f32(w, h, spp)
        assert_bits(np.load(tmp_path / ("%d.npy" % i)), ref, "shape %d case %d" % (shape, i))


@pytest.mark.gpu
def test_f32_error_codes(rt, gpu_scene8):
    import torch
    L, w, h = rt.lib(), 64, 32
    dev = torch.device("cuda", gpu_scene8.device())
    t = torch.zeros(w * h * 4 + 8, dtype=torch.float32, device=dev)
    arr = (rt.C.c_void_p * 1)(gpu_scene8.handle)

    def rows(ptr, pitch=0):
        return L.rt_render_rows_f32(gpu_scene8.handle, None, w, h, 1, 0, 1, h, ptr, pitch, None, None)

    assert rows(None) == rt.RT_ERR_INVALID                           # no output
    assert rows(t.data_ptr() + 4) == rt.RT_ERR_INVALID               # device output not 16-byte aligned
    assert rows(t.data_ptr() + 8) == rt.RT_ERR_INVALID
    assert rows(t.data_ptr(), w * 16 + 4) == rt.RT_ERR_INVALID       # pitch not a multiple of 16
    assert rows(t.data_ptr(), w * 16 - 16) == rt.RT_ERR_INVALID      # pitch shorter than a row
    assert rows(t.data_ptr()) == rt.RT_OK
    assert L.rt_render_rows_f32(None, None, w, h, 1, 0, 1, h, t.data_ptr(), 0, None, None) == rt.RT_ERR_INVALID
    assert L.rt_render_rows_f32(gpu_scene8.handle, None, w, h, 1, 0, 1, h + 1, t.data_ptr(), 0, None, None) \
        == rt.RT_ERR_INVALID                                         # rows leave the image
    multi = L.rt_render_frame_multi_f32
    assert multi(arr, 1, None, w, h, 1, t.data_ptr(), w * h * 16 - 1, None) == rt.RT_ERR_BUFFER
    assert multi(arr, 1, None, w, h, 1, None, w * h * 16, None) == rt.RT_ERR_INVALID
    assert multi(arr, 1, None, w, h, 1, t.data_ptr() + 4, w * h * 16, None) == rt.RT_ERR_INVALID
    assert multi(arr, 0, None, w, h, 1, t.data_ptr(), w * h * 16, None) == rt.RT_ERR_INVALID
    assert multi(arr, 1, None, 0, h, 1, t.data_ptr(), w * h * 16, None) == rt.RT_ERR_INVALID
    assert multi(arr, 1, None, w, h, 1, t.data_ptr(), w * h * 16, None) == rt.RT_OK
    torch.cuda.synchronize(dev)


@pytest.mark.gpu
def test_f32_two_gpus_equal_one(rt, f32_scene8):
    if rt.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    import torch
    scenes = []
    for g in range(2):
        rt.set_device(g)
        scenes.append(rt.Scene())
    rt.set_device(0)
    for w, h, spp in ((1000, 333, 2), (640, 480, 1)):
        o = rt.RenderOptions(w, h, spp)
        one = rt.Renderer.render_f32(o, scenes[0])
        ref, _ = f32_scene8.render_f32(w, h, spp)
        assert_bits(one, ref, "one GPU")
        two, st = rt.Renderer.render_f32(o, scenes, want_stats=True)
        assert st.gpus == 2
        assert_bits(two, one, "two GPUs, host output")
        d = torch.empty((h, w, 4), dtype=torch.float32, device="cuda:0")
        rt.Renderer.render_f32(o, scenes, out_ptr=d.data_ptr())
        assert_bits(d.cpu().numpy(), one, "two GPUs, device output")
    for s in scenes:
        s.close()


@pytest.mark.gpu
def test_cli_pfm_writes_the_oracle_floats(rtrace, tmp_path):
    """C1 as `rtrace --format pfm`: header + the oracle's float RGB rows, bottom row first; its values re-quantised
    are the reference's shipped image."""
    w, h, spp = GOLD["width"], GOLD["height"], GOLD["spp"]
    r = run(rtrace, "--format=pfm", "--samples-per-pixel=%d" % spp, "--width=%d" % w, "--height=%d" % h, "--stats", "out.pfm",
            cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout == b"", r.stderr
    assert b"kernel" in r.stderr
    ref, _ = _oracle_f32.Scene().render_f32(w, h, spp)
    data = (tmp_path / "out.pfm").read_bytes()
    assert data == pfm_bytes(ref)
    rgb = quantise(np.frombuffer(data[len(b"PF\n1024 768\n-1.0\n"):], "<f4").reshape(h, w, 3)[::-1])
    assert hashlib.sha256(np.ascontiguousarray(rgb).tobytes()).hexdigest() == GOLD["rgb_sha256"]


@pytest.mark.gpu
def test_cli_pfm_frames_and_stdout(rtrace, oracle, tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    w, h, spp, n = 160, 90, 2, 3
    s = _oracle_f32.Scene()
    refs = [s.render_f32(w, h, spp, camera=oracle.make_camera(*bench.orbit_basis(f, n)))[0] for f in range(n)]
    r = run(rtrace, "--format=pfm", "--frames=%d" % n, "--width=%d" % w, "--height=%d" % h,
            "--samples-per-pixel=%d" % spp, "s.pfm", cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr
    assert sorted(p.name for p in tmp_path.iterdir()) == ["s.0000.pfm", "s.0001.pfm", "s.0002.pfm"]
    for f in range(n):
        assert (tmp_path / ("s.%04d.pfm" % f)).read_bytes() == pfm_bytes(refs[f]), f
    r = run(rtrace, "--format=pfm", "--frames=%d" % n, "--width=%d" % w, "--height=%d" % h,
            "--samples-per-pixel=%d" % spp, "-", cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout == b"".join(pfm_bytes(x) for x in refs)
    r = run(rtrace, "--format=pfm", "--width=%d" % w, "--height=%d" % h, "--samples-per-pixel=%d" % spp, "-")
    assert r.returncode == 0 and r.stdout == pfm_bytes(refs[0])
