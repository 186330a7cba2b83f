"""Geometry output (AOVs): rt_render_rows_aov, rt_render_frame_multi_aov and `rtrace --format pfm --aov`.

An AOV pixel is eight f32 {nx, ny, nz, coverage, distance, px, py, pz} (include/rtrace.h "geometry output"): over the
pixel's primary samples that hit, the box-filtered unit normal, the covered fraction, and the nearest hit's distance
and point.  The CPU part ties the AOV oracle (tests/_oracle_aov.cpp) to the pinned oracle's kinds and ray hits
(tests/_aov_ref.py) and checks the PFM writers and the command line; the GPU part checks the kernels (PHASED's AOV
store and the LANE kernel) against the oracle bit for bit."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _aov_ref
import _cameras
import _oracle_aov
import _oracle_f32
from _aov_ref import assert_bits

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "target", "release", "rtrace")
SELFTEST = os.path.join(ROOT, "target", "release", "rtrace_selftest")
AOV_GOLD = json.load(open(os.path.join(HERE, "golden", "oracle_aov.json")))
CAMS = _cameras.named_cameras()
AOV_FILES = (("normal", slice(0, 3)), ("coverage", slice(3, 4)), ("distance", slice(4, 5)), ("position", slice(5, 8)))


def aov_sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<f4").tobytes()).hexdigest()


def pfm_bytes(img):
    """A PFM of (h, w, 3) or (h, w, 1) floats: "PF" / "Pf", size, -1.0, rows bottom-up, little-endian."""
    h, w, c = img.shape
    return (b"PF" if c == 3 else b"Pf") + b"\n%d %d\n-1.0\n" % (w, h) + \
        np.ascontiguousarray(img[::-1], dtype="<f4").tobytes()


def run(cmd, *args, cwd=None, timeout=300):
    return subprocess.run([cmd] + list(args), capture_output=True, cwd=cwd, timeout=timeout)


@pytest.fixture(scope="module")
def rtrace():
    if not (os.path.exists(BIN) and os.path.exists(SELFTEST)):
        subprocess.check_call(["make", "-s", "-C", ROOT, "rtrace"])
    return BIN


@pytest.fixture(scope="module")
def aov_scene8():
    """The default scene (level 8) in the AOV oracle."""
    return _oracle_aov.Scene()


def named(name):
    eye, b = CAMS[name]
    return eye, b


# ---- CPU: the AOV oracle against the pinned one, the PFM writers, the command line --------------------------------
@pytest.mark.parametrize("w,h,spp,level", [(64, 48, 1, 2), (33, 7, 2, 8), (40, 30, 3, 5), (97, 61, 4, 9),
                                          (24, 16, 5, 3), (20, 12, 6, 8), (17, 9, 7, 6), (16, 8, 8, 8),
                                          (12, 8, 9, 4), (1, 1, 1, 8), (32, 18, 1, 10), (24, 12, 2, 11),
                                          (16, 9, 1, 12)])
def test_aov_oracle_is_the_pinned_oracles_geometry(oracle, w, h, spp, level):
    a = _oracle_aov.Scene(level=level).render_aov(w, h, spp)
    pinned = oracle.Scene(level=level)
    _aov_ref.check_rows_coverage(a, pinned, w, h, spp, range(h))
    _aov_ref.check_rows_against_traced_rays(a, pinned, w, h, spp, range(h), pinned.eye())
    miss = a[..., 3] == 0
    assert (a[..., 4][miss] == np.inf).all() and (a[..., 4][~miss] < np.inf).all()
    assert not np.isnan(a).any()


@pytest.mark.parametrize("frame", [0, 7, 41, 88])
def test_aov_oracle_orbit_cameras_and_rows(oracle, frame):
    sys.path.insert(0, ROOT)
    import bench
    eye, right, up, fwd = bench.orbit_basis(frame)
    cam = oracle.make_camera(eye, right, up, fwd)
    s, pinned = _oracle_aov.Scene(level=8), oracle.Scene(level=8)
    w, h, spp = 120, 90, 2
    a = s.render_aov(w, h, spp, camera=cam)
    _aov_ref.check_rows_coverage(a, pinned, w, h, spp, range(h), cam)
    _aov_ref.check_rows_against_traced_rays(a, pinned, w, h, spp, range(h), eye, np.array([right, up, fwd], np.float32))
    assert_bits(s.render_aov(w, h, spp, row_start=1, row_stride=3, camera=cam), a[1::3], "rows 1, 4, 7, ...")


@pytest.mark.parametrize("name", ["general", "roll30", "off_light"])
def test_aov_oracle_general_camera_bases(oracle, name):
    eye, b = named(name)
    cam = oracle.make_camera(eye, b[0], b[1], b[2])
    w, h, spp = 96, 54, 3
    a = _oracle_aov.Scene().render_aov(w, h, spp, camera=cam)
    pinned = oracle.Scene()
    _aov_ref.check_rows_coverage(a, pinned, w, h, spp, range(h), cam)
    _aov_ref.check_rows_against_traced_rays(a, pinned, w, h, spp, range(h), eye, b)
    assert (a[..., 3] > 0).any()


def test_aov_c1_matches_fixture(aov_scene8):
    c1 = [c for c in AOV_GOLD["cases"] if (c["width"], c["height"], c["spp"], c["level"]) == (1024, 768, 4, 8)]
    assert len(c1) == 1
    assert aov_sha(aov_scene8.render_aov(1024, 768, 4)) == c1[0]["aov_sha256"]


def test_pfm_writers_layout(rtrace, tmp_path):
    """write_pfm (host/render.hpp) on the selftest's synthetic 3x2 frame: the colour PFM and the greyscale Pf of
    component 3, both little-endian, bottom row first, the source pitch followed."""
    r = run(SELFTEST, "pfm", str(tmp_path / "t.pfm"))
    assert r.returncode == 0 and b"ok pfm" in r.stdout, r.stderr
    px = (np.arange(24, dtype=np.float32) / np.float32(7.0)).reshape(2, 3, 4)
    assert (tmp_path / "t.pfm").read_bytes() == pfm_bytes(px[..., :3])
    grey = (tmp_path / "t.pfm.grey.pfm").read_bytes()
    assert grey == pfm_bytes(px[..., 3:4])
    assert grey.startswith(b"Pf\n3 2\n-1.0\n") and len(grey) == 12 + 2 * 3 * 4
    assert np.frombuffer(grey[12:16], "<f4")[0] == px[1, 0, 3]   # the bottom row comes first


def test_cli_aov_arguments(rtrace, tmp_path):
    for args, flag in ((["--aov", "o.tga"], b"'--format pfm'"), (["--format=tga", "--aov", "o.tga"], b"'--format pfm'"),
                       (["--format=png", "--aov", "o.png"], b"'--format pfm'"), (["--format=pfm", "--aov", "-"], b"'-'"),
                       (["--format=pfm", "--aov", "--buckets", "o.pfm"], b"--buckets"),
                       (["--format=pfm", "--aov", "--preview=4", "o.pfm"], b"--preview")):
        r = run(rtrace, *args, cwd=str(tmp_path))
        assert r.returncode == 1 and flag in r.stderr, (args, r.stderr)
    r = run(rtrace, "--format=pfm", "--aov", "picture.tga", cwd=str(tmp_path))
    assert r.returncode == 0 and b"must have the pfm extension" in r.stdout
    assert not list(tmp_path.iterdir())
    h = run(rtrace, "--help").stdout
    assert b"--aov" in h and b".normal.pfm" in h


# ---- GPU ----------------------------------------------------------------------------------------------------------
def expected_variant(rt, scene, w, h, spp, variant, camera=None):
    """The float output's variant rule (test_f32.py): LANE for a forced LANE or WARP; for a forced TILE or PHASED
    what a forced PHASED runs; AUTO: PHASED where RGBA8 runs TILE or PHASED."""
    if variant in (rt.VARIANT_LANE, rt.VARIANT_WARP):
        return rt.VARIANT_LANE
    rt.set_variant(rt.VARIANT_PHASED if variant != rt.VARIANT_AUTO else rt.VARIANT_AUTO)
    try:
        _, st = rt.Renderer.render(rt.RenderOptions(w, h, spp), scene, camera=camera, want_stats=True)
    finally:
        rt.set_variant(rt.VARIANT_AUTO)
    return rt.VARIANT_LANE if st.variant_used == rt.VARIANT_LANE else rt.VARIANT_PHASED


ALL_VARIANTS = ("VARIANT_AUTO", "VARIANT_LANE", "VARIANT_WARP", "VARIANT_TILE", "VARIANT_PHASED")


def render_aov_as(rt, variant, options, scene, camera=None):
    rt.set_variant(variant)
    try:
        return rt.Renderer.render_aov(options, scene, camera=camera, want_stats=True)
    finally:
        rt.set_variant(rt.VARIANT_AUTO)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,spp,level", [(64, 128, 2, 8), (160, 120, 1, 8), (160, 120, 3, 8), (200, 150, 4, 5),
                                          (97, 61, 2, 9), (256, 144, 1, 10), (33, 7, 1, 8), (1, 1, 1, 8), (8, 4, 5, 2),
                                          (320, 180, 5, 7), (200, 120, 6, 8), (131, 77, 7, 6), (256, 144, 8, 8),
                                          (40, 30, 9, 5), (96, 54, 1, 11), (48, 27, 2, 12)])
def test_aov_frame_matches_oracle(rt, w, h, spp, level):
    gs, os_ = rt.Scene(level=level), _oracle_aov.Scene(level=level)
    ref = os_.render_aov(w, h, spp)
    for name in ALL_VARIANTS:
        v = getattr(rt, name)
        want = expected_variant(rt, gs, w, h, spp, v)
        img, st = render_aov_as(rt, v, rt.RenderOptions(w, h, spp), gs)
        assert_bits(img, ref, "%s %dx%d spp %d L%d" % (name, w, h, spp, level))
        assert st.variant_used == want, (name, st.variant_used, want)
        assert st.kernel_launches == (3 if want == rt.VARIANT_PHASED else 1)   # no shadow cull, no shading
        assert (st.primary_rays, st.shadow_rays) == (w * h * spp * spp, 0)
    gs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h,spp", [("general", 224, 126, 1), ("general", 161, 93, 4), ("roll30", 224, 126, 2),
                                          ("off_light", 160, 90, 8), ("sideways", 1280, 720, 1),
                                          ("along_light", 1280, 720, 2)])
def test_aov_general_camera_bases(rt, name, w, h, spp):
    eye, b = named(name)
    gs, os_ = rt.Scene(), _oracle_aov.Scene()
    import _oracle
    ref = os_.render_aov(w, h, spp, camera=_oracle.make_camera(eye, b[0], b[1], b[2]))
    cam = rt.make_camera(eye, b[0], b[1], b[2])
    for v in (rt.VARIANT_AUTO, rt.VARIANT_PHASED, rt.VARIANT_LANE):
        img, st = render_aov_as(rt, v, rt.RenderOptions(w, h, spp), gs, cam)
        assert st.variant_used == (rt.VARIANT_LANE if v == rt.VARIANT_LANE else expected_variant(rt, gs, w, h, spp, v, cam))
        assert_bits(img, ref, "%s %dx%d spp %d variant %d" % (name, w, h, spp, v))
    gs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", AOV_GOLD["cases"],
                         ids=lambda c: "%dx%d_spp%d_L%d" % (c["width"], c["height"], c["spp"], c["level"]))
def test_aov_baseline_frames_match_fixture(rt, case):
    """Every BASELINE configuration at full size on PHASED (what AUTO runs there) and on the forced LANE kernel."""
    gs = rt.Scene(level=case["level"])
    o = rt.RenderOptions(case["width"], case["height"], case["spp"])
    for v in (rt.VARIANT_AUTO, rt.VARIANT_LANE):
        img, st = render_aov_as(rt, v, o, gs)
        assert st.variant_used == (rt.VARIANT_PHASED if v == rt.VARIANT_AUTO else rt.VARIANT_LANE)
        assert aov_sha(img) == case["aov_sha256"], v
    gs.close()


@pytest.mark.gpu
def test_aov_c5_orbit_frames_match_fixture(rt):
    cases = AOV_GOLD["c5_cases"]
    gs = rt.Scene(level=cases[0]["level"])
    for c in cases:
        o = rt.RenderOptions(c["width"], c["height"], c["spp"])
        img, st = rt.Renderer.render_aov(o, gs, camera=rt.orbit_camera(c["frame"], c["n_frames"]), want_stats=True)
        assert st.variant_used == rt.VARIANT_PHASED
        assert aov_sha(img) == c["aov_sha256"], "orbit frame %d" % c["frame"]
    gs.close()


@pytest.mark.gpu
def test_aov_fallbacks_run_lane_and_match_oracle(rt, oracle):
    light = np.array([-1.0, -3.0, 2.0], np.float32)
    light /= np.float32(np.sqrt(np.float32((light * light).sum())))
    sph = np.array([[0, -1, 0, 2], [-0.6, -1, 0, 0.5], [0.6, -1, 0.3, 0.5], [0, -0.2, 0, 0.4]], np.float32)
    skip = np.array([4, 2, 3, 4], np.uint32)
    cases = [("level 11", lambda: (rt.Scene(level=11), _oracle_aov.Scene(level=11)), (96, 54, 1)),
             ("level 12", lambda: (rt.Scene(level=12), _oracle_aov.Scene(level=12)), (48, 27, 2)),
             ("hand-built group", lambda: (rt.Scene.from_nodes(sph, skip, light, (0, 0, -4)),
                                           _oracle_aov.Scene.from_nodes(sph, skip, light, (0, 0, -4))), (80, 60, 2)),
             ("spp 9", lambda: (rt.Scene(), _oracle_aov.Scene()), (40, 30, 9)),
             ("eye inside the root bound", lambda: (rt.Scene(eye=(0.0, -0.6, -0.3)),
                                                    _oracle_aov.Scene(eye=(0.0, -0.6, -0.3))), (64, 48, 2))]
    for what, make, (w, h, spp) in cases:
        gs, os_ = make()
        ref = os_.render_aov(w, h, spp)
        for name in ("VARIANT_AUTO", "VARIANT_PHASED", "VARIANT_TILE"):
            img, st = render_aov_as(rt, getattr(rt, name), rt.RenderOptions(w, h, spp), gs)
            assert st.variant_used == rt.VARIANT_LANE, (what, name)
            assert_bits(img, ref, "%s (%s)" % (what, name))
        gs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("spp", [1, 2, 4, 8])
def test_aov_pool_overflow_walk(rt, spp):
    """A tiny candidate pool (RTRACE_POOL_UNITS) sends cull tiles to K2's per-lane walk; the AOV store reads the
    winners that walk wrote."""
    w, h = 320, 180
    gs = rt.Scene(level=9)
    ref = _oracle_aov.Scene(level=9).render_aov(w, h, spp)
    try:
        for units in ("64", "4096", "65536"):
            os.environ["RTRACE_POOL_UNITS"] = units
            img, st = render_aov_as(rt, rt.VARIANT_PHASED, rt.RenderOptions(w, h, spp), gs)
            assert st.variant_used == rt.VARIANT_PHASED
            assert_bits(img, ref, "spp %d pool of %s units" % (spp, units))
    finally:
        os.environ.pop("RTRACE_POOL_UNITS", None)
        gs.close()


SHAPE_SCRIPT = r"""
import json, sys
import numpy as np
import rtrace_b200 as rt
cases = json.loads(sys.argv[1])
scene = rt.Scene()
used = {}
for i, (variant, w, h, spp) in enumerate(cases):
    rt.set_variant(variant)
    img, st = rt.Renderer.render_aov(rt.RenderOptions(w, h, spp), scene, want_stats=True)
    np.save("%s/%d.npy" % (sys.argv[2], i), img)
    used[i] = int(st.variant_used)
json.dump(used, open(sys.argv[2] + "/used.json", "w"))
scene.close()
"""


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [0, 1, 2, 3, 4, 5, 6])
def test_aov_every_tile_shape(rt, aov_scene8, shape, tmp_path):
    """RTRACE_TILE_SHAPE (read once per process, so each shape runs in a process of its own) forces every spp-1
    tile shape of PHASED, and the 4x4 shape of spp 2 and 4 where it exists."""
    cases = [(rt.VARIANT_PHASED, 173, 91, 1), (rt.VARIANT_PHASED, 1920, 1080, 1), (rt.VARIANT_PHASED, 130, 70, 2),
             (rt.VARIANT_PHASED, 96, 64, 4), (rt.VARIANT_TILE, 61, 47, 1)]
    env = dict(os.environ, RTRACE_TILE_SHAPE=str(shape),
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "rust-tracer_b200"), HERE]))
    subprocess.run([sys.executable, "-c", SHAPE_SCRIPT, json.dumps(cases), str(tmp_path)], env=env, check=True,
                   timeout=900)
    used = json.loads((tmp_path / "used.json").read_text())
    for i, (variant, w, h, spp) in enumerate(cases):
        assert used[str(i)] == rt.VARIANT_PHASED, (i, used[str(i)])
        assert_bits(np.load(tmp_path / ("%d.npy" % i)), aov_scene8.render_aov(w, h, spp), "shape %d case %d" % (shape, i))


@pytest.mark.gpu
def test_aov_rows_pitch_and_host_memory(rt, aov_scene8, gpu_scene8):
    """Strided rows, a pitch wider than the row, pageable and pinned host memory."""
    import torch
    w, h, spp = 200, 150, 2
    o = rt.RenderOptions(w, h, spp)
    full = aov_scene8.render_aov(w, h, spp)
    for variant in (rt.VARIANT_AUTO, rt.VARIANT_PHASED, rt.VARIANT_LANE):
        rt.set_variant(variant)
        try:
            rows = rt.Renderer.render_rows_aov(o, gpu_scene8, row_start=2, row_stride=3)
            assert_bits(rows, full[2::3], "rows 2, 5, 8, ...")
            pitch = w * 32 + 48
            buf = np.full((h, pitch // 4), np.float32(-7.0), np.float32)   # pageable, padded rows
            rt.Renderer.render_rows_aov(o, gpu_scene8, out_ptr=buf.ctypes.data, pitch=pitch)
            assert_bits(np.ascontiguousarray(buf[:, :w * 8]).reshape(h, w, 8), full, "pitched host rows")
            assert (buf[:, w * 8:] == np.float32(-7.0)).all()   # the padding is left alone
            pinned = torch.empty((h, w, 8), dtype=torch.float32, pin_memory=True)
            rt.Renderer.render_rows_aov(o, gpu_scene8, out_ptr=pinned.data_ptr())
            assert_bits(pinned.numpy(), full, "pinned host frame")
        finally:
            rt.set_variant(rt.VARIANT_AUTO)


@pytest.mark.gpu
def test_aov_into_a_torch_cuda_tensor(rt, aov_scene8, gpu_scene8):
    """Device output on torch's current stream: asynchronous, ordered with torch's own work on that stream; a pitch
    that is a multiple of 16 but not of 32."""
    import torch
    w, h, spp = 320, 240, 4
    o = rt.RenderOptions(w, h, spp)
    ref = aov_scene8.render_aov(w, h, spp)
    dev = torch.device("cuda", gpu_scene8.device())
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.device(dev), torch.cuda.stream(side):
        t = torch.full((h, w, 8), float("nan"), dtype=torch.float32, device=dev)
        rt.Renderer.render_rows_aov(o, gpu_scene8, out_ptr=t.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        covered = t[..., 3].sum()   # queued behind the render on the same stream
        pitched = torch.full((h, w * 8 + 4), -1.0, dtype=torch.float32, device=dev)
        rt.Renderer.render_rows_aov(o, gpu_scene8, out_ptr=pitched.data_ptr(), pitch=(w * 8 + 4) * 4,
                                    stream=torch.cuda.current_stream().cuda_stream)
        got, got_pitched, covered = t.cpu().numpy(), pitched.cpu().numpy(), float(covered.cpu())
    assert_bits(got, ref, "torch tensor")
    assert_bits(np.ascontiguousarray(got_pitched[:, :w * 8]).reshape(h, w, 8), ref, "pitched torch tensor")
    assert (got_pitched[:, w * 8:] == -1.0).all()
    assert covered == pytest.approx(float(ref[..., 3].sum(dtype=np.float64)), rel=1e-5)
    dframe = torch.empty((h, w, 8), dtype=torch.float32, device=dev)
    assert rt.Renderer.render_aov(o, gpu_scene8, out_ptr=dframe.data_ptr()) is None
    assert_bits(dframe.cpu().numpy(), ref, "rt_render_frame_multi_aov, device output")


@pytest.mark.gpu
def test_aov_error_codes(rt, gpu_scene8):
    import torch
    L, w, h = rt.lib(), 64, 32
    dev = torch.device("cuda", gpu_scene8.device())
    t = torch.zeros(w * h * 8 + 8, dtype=torch.float32, device=dev)
    arr = (rt.C.c_void_p * 1)(gpu_scene8.handle)

    def rows(ptr, pitch=0):
        return L.rt_render_rows_aov(gpu_scene8.handle, None, w, h, 1, 0, 1, h, ptr, pitch, None, None)

    assert rows(None) == rt.RT_ERR_INVALID                           # no output
    assert rows(t.data_ptr() + 4) == rt.RT_ERR_INVALID               # device output not 16-byte aligned
    assert rows(t.data_ptr() + 8) == rt.RT_ERR_INVALID
    assert rows(t.data_ptr(), w * 32 + 8) == rt.RT_ERR_INVALID       # pitch not a multiple of 16
    assert rows(t.data_ptr(), w * 32 - 16) == rt.RT_ERR_INVALID      # pitch shorter than a row
    assert L.rt_render_rows_aov(gpu_scene8.handle, None, w, h, 1, 0, 1, h - 1, t.data_ptr(), w * 32 + 16, None, None) \
        == rt.RT_OK                                                  # a pitch of 16 * odd bytes is accepted
    assert rows(t.data_ptr() + 16) == rt.RT_OK                       # 16-byte aligned is enough
    assert rows(t.data_ptr()) == rt.RT_OK
    assert L.rt_render_rows_aov(None, None, w, h, 1, 0, 1, h, t.data_ptr(), 0, None, None) == rt.RT_ERR_INVALID
    assert L.rt_render_rows_aov(gpu_scene8.handle, None, w, h, 1, 0, 1, h + 1, t.data_ptr(), 0, None, None) \
        == rt.RT_ERR_INVALID                                         # rows leave the image
    multi = L.rt_render_frame_multi_aov
    assert multi(arr, 1, None, w, h, 1, t.data_ptr(), w * h * 32 - 1, None) == rt.RT_ERR_BUFFER
    assert multi(arr, 1, None, w, h, 1, None, w * h * 32, None) == rt.RT_ERR_INVALID
    assert multi(arr, 1, None, w, h, 1, t.data_ptr() + 4, w * h * 32, None) == rt.RT_ERR_INVALID
    assert multi(arr, 0, None, w, h, 1, t.data_ptr(), w * h * 32, None) == rt.RT_ERR_INVALID
    assert multi(arr, 1, None, 0, h, 1, t.data_ptr(), w * h * 32, None) == rt.RT_ERR_INVALID
    assert multi(arr, 1, None, w, h, 1, t.data_ptr(), w * h * 32, None) == rt.RT_OK
    torch.cuda.synchronize(dev)


@pytest.mark.gpu
def test_aov_two_gpus_equal_one(rt, aov_scene8):
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
        one = rt.Renderer.render_aov(o, scenes[0])
        assert_bits(one, aov_scene8.render_aov(w, h, spp), "one GPU")
        two, st = rt.Renderer.render_aov(o, scenes, want_stats=True)
        assert st.gpus == 2 and st.shadow_rays == 0
        assert_bits(two, one, "two GPUs, host output")
        d = torch.empty((h, w, 8), dtype=torch.float32, device="cuda:0")
        rt.Renderer.render_aov(o, scenes, out_ptr=d.data_ptr())
        assert_bits(d.cpu().numpy(), one, "two GPUs, device output")
    for s in scenes:
        s.close()


def expected_files(aov, colour):
    """The five files of `--format pfm --aov` for one frame."""
    files = {"": pfm_bytes(colour[..., :3])}
    for name, sl in AOV_FILES:
        files["." + name] = pfm_bytes(aov[..., sl])
    return files


@pytest.mark.gpu
def test_cli_aov_writes_five_files(rtrace, tmp_path):
    """`rtrace --format pfm --aov` at 1024x768, 4x4 samples: out.pfm byte-identical to the run without --aov, and
    the four AOV files the oracle's values."""
    w, h, spp = 1024, 768, 4
    args = ["--format=pfm", "--width=%d" % w, "--height=%d" % h, "--samples-per-pixel=%d" % spp]
    (tmp_path / "plain").mkdir()
    r = run(rtrace, *args, "out.pfm", cwd=str(tmp_path / "plain"))
    assert r.returncode == 0, r.stderr
    r = run(rtrace, *args, "--aov", "--stats", "out.pfm", cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout == b"" and b"kernel" in r.stderr, r.stderr
    names = ["out.pfm"] + ["out.%s.pfm" % n for n, _ in AOV_FILES]
    assert sorted(p.name for p in tmp_path.iterdir() if p.is_file()) == sorted(names)
    assert (tmp_path / "out.pfm").read_bytes() == (tmp_path / "plain" / "out.pfm").read_bytes()
    aov = _oracle_aov.Scene().render_aov(w, h, spp)
    for name, sl in AOV_FILES:
        assert (tmp_path / ("out.%s.pfm" % name)).read_bytes() == pfm_bytes(aov[..., sl]), name


@pytest.mark.gpu
def test_cli_aov_frames_and_gpus(rt, rtrace, oracle, tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    w, h, spp, n = 160, 90, 2, 3
    s, colour = _oracle_aov.Scene(), _oracle_f32.Scene()
    cams = [oracle.make_camera(*bench.orbit_basis(f, n)) for f in range(n)]
    want = {}
    for f in range(n):
        for suffix, data in expected_files(s.render_aov(w, h, spp, camera=cams[f]),
                                           colour.render_f32(w, h, spp, camera=cams[f])[0]).items():
            want["s.%04d%s.pfm" % (f, suffix)] = data
    for gpus in sorted({1, min(2, rt.device_count())}):
        d = tmp_path / ("g%d" % gpus)
        d.mkdir()
        r = run(rtrace, "--format=pfm", "--aov", "--frames=%d" % n, "--gpus=%d" % gpus, "--width=%d" % w,
                "--height=%d" % h, "--samples-per-pixel=%d" % spp, "s.pfm", cwd=str(d))
        assert r.returncode == 0, r.stderr
        assert sorted(p.name for p in d.iterdir()) == sorted(want)
        for name, data in want.items():
            assert (d / name).read_bytes() == data, (gpus, name)
