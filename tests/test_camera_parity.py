"""Rendering under general camera bases, and hand-built trees, against the CPU oracle.

The orbit camera is a rotation about y: four of its nine basis entries are 0 and one is 1, so an error in a row of
the camera rotation (primary_dir, slot_dir, the packed slot_dir2, the cull cone's axis, PHASED's screen_box) passes
every orbit frame.  The named cameras of tests/_cameras.py have no zero entry (most of them), one is mirrored, two
put the primary beams along / nearly along the shadow rays and one sees spheres behind its image plane.  Every
variant and every entry point that takes a camera must return the oracle's bytes for them, and the fast variants
must really run (rt_stats.variant_used).

The second half renders trees built with rt_scene_create_from_nodes: overlapping siblings, children poking out of
their bound, duplicate spheres, a deep chain, a root of leaves only and an eye inside a group bound -- the
per-lane walks' pruning has otherwise only seen the pyramid."""
import os

import numpy as np
import pytest

import _cameras

pytestmark = pytest.mark.gpu

CAMS = _cameras.named_cameras()
F = np.float32


def rt_camera(rt, name_or_pair):
    eye, b = CAMS[name_or_pair] if isinstance(name_or_pair, str) else name_or_pair
    return rt.make_camera(eye, b[0], b[1], b[2])


def oracle_camera(oracle, name_or_pair):
    eye, b = CAMS[name_or_pair] if isinstance(name_or_pair, str) else name_or_pair
    return oracle.make_camera(eye, b[0], b[1], b[2])


def assert_same(gpu, ref, what=""):
    if not np.array_equal(gpu, ref):
        diff = np.abs(gpu.astype(np.int16) - ref.astype(np.int16))
        diff = diff.max(axis=-1) if diff.ndim == 3 else diff
        ys, xs = np.nonzero(diff)[:2]
        raise AssertionError("%s: %d of %d pixels differ (max %d), first at row %d col %d: gpu %s ref %s" % (
            what, len(ys), diff.size, diff.max(), ys[0], xs[0], gpu[ys[0], xs[0]], ref[ys[0], xs[0]]))


def render_variant(rt, variant, options, scene, camera, kinds=True):
    rt.set_variant(variant)
    try:
        return rt.Renderer.render_rows(options, scene, camera=camera, kinds=kinds, want_stats=True)
    finally:
        rt.set_variant(rt.VARIANT_AUTO)


@pytest.fixture(scope="module")
def scenes(rt, oracle):
    return rt.Scene(), oracle.Scene()


def test_named_cameras_are_general_and_within_the_tolerance():
    for name, (eye, b) in CAMS.items():
        bd = b.astype(np.float64)
        assert np.abs(bd @ bd.T - np.eye(3)).max() <= 1e-6, name
        assert _cameras.orthonormal32(b, 1e-6), name
    for name in _cameras.FULL_BASIS:
        assert np.abs(CAMS[name][1]).min() >= 0.05, name


# (camera, width, height, spp): TILE runs spp 1 .. 4, PHASED spp 1 .. 8, each with a full basis somewhere
CASES = [("pitched_down", 224, 126, 1), ("from_below", 224, 126, 2), ("roll30", 224, 126, 3), ("roll90", 224, 126, 4),
         ("general", 224, 126, 4), ("general", 160, 90, 5), ("mirrored", 224, 126, 2), ("mirrored", 160, 90, 6),
         ("along_light", 224, 126, 1), ("along_light", 160, 90, 7), ("off_light", 224, 126, 3),
         ("off_light", 160, 90, 8), ("sideways", 224, 126, 2), ("sideways", 160, 90, 4)]


@pytest.mark.parametrize("name,w,h,spp", CASES, ids=["%s-%dx%d-spp%d" % c for c in CASES])
def test_every_variant_matches_oracle_under_named_camera(rt, oracle, scenes, name, w, h, spp):
    gs, os_ = scenes
    ref, okinds, ctr = os_.render_region(w, h, spp, 0, 0, w, h, camera=oracle_camera(oracle, name), kinds=True)
    cam = rt_camera(rt, name)
    variants = [rt.VARIANT_LANE, rt.VARIANT_WARP, rt.VARIANT_PHASED] + ([rt.VARIANT_TILE] if spp <= 4 else [])
    for v in variants:
        img, kinds, st = render_variant(rt, v, rt.RenderOptions(w, h, spp), gs, cam)
        assert st.variant_used == v, "%s: variant %d fell back to %d" % (name, v, st.variant_used)
        assert np.array_equal(kinds, okinds), "%s spp %d: per-sample mask differs for variant %d" % (name, spp, v)
        assert_same(img, ref, "%s spp %d variant %d" % (name, spp, v))
    assert gs.count_rays(w, h, spp, camera=cam) == (ctr.primary_rays, ctr.shadow_rays)
    assert ctr.primary_hits > 0


BIG = [("general", 1280, 720, 1), ("along_light", 1280, 720, 2), ("off_light", 1600, 900, 1), ("sideways", 1280, 720, 1)]


@pytest.mark.parametrize("name,w,h,spp", BIG, ids=["%s-%dx%d-spp%d" % c for c in BIG])
def test_candidate_list_variants_in_the_phased_regime(rt, oracle, scenes, name, w, h, spp):
    """Tiles small against the spheres: the image-space boxes and the shadow discs prune for real."""
    gs, os_ = scenes
    ref, ctr = os_.render(w, h, spp, camera=oracle_camera(oracle, name))
    cam = rt_camera(rt, name)
    for v in (rt.VARIANT_TILE, rt.VARIANT_PHASED):
        img, st = render_variant(rt, v, rt.RenderOptions(w, h, spp), gs, cam, kinds=False)
        assert st.variant_used == v
        assert_same(img, ref, "%s %dx%d spp %d variant %d" % (name, w, h, spp, v))
    assert gs.count_rays(w, h, spp, camera=cam) == (ctr.primary_rays, ctr.shadow_rays)


@pytest.mark.parametrize("w,h,spp", [(4000, 24, 2), (24, 3000, 1)])
def test_extreme_aspect_ratios(rt, oracle, scenes, w, h, spp):
    """A 24-pixel-wide frame 3000 rows tall has a vertical field of view close to 180 degrees: rays almost
    perpendicular to `forward`, cull cones at grazing angles."""
    gs, os_ = scenes
    ref, okinds, ctr = os_.render_region(w, h, spp, 0, 0, w, h, camera=oracle_camera(oracle, "general"), kinds=True)
    cam = rt_camera(rt, "general")
    for v in (rt.VARIANT_TILE, rt.VARIANT_PHASED):
        img, kinds, st = render_variant(rt, v, rt.RenderOptions(w, h, spp), gs, cam)
        assert st.variant_used == v
        assert np.array_equal(kinds, okinds), "%dx%d variant %d: mask differs" % (w, h, v)
        assert_same(img, ref, "%dx%d variant %d" % (w, h, v))
    assert ctr.primary_hits > 0
    assert gs.count_rays(w, h, spp, camera=cam) == (ctr.primary_rays, ctr.shadow_rays)


@pytest.mark.parametrize("name,step", [("general", 1), ("mirrored", 5), ("off_light", 16)])
def test_preview_under_named_camera(rt, oracle, scenes, name, step):
    gs, os_ = scenes
    w, h = 257, 143
    full, _ = os_.render(w, h, 1, camera=oracle_camera(oracle, name))
    ys, xs = (np.arange(h) // step) * step, (np.arange(w) // step) * step
    got = rt.Renderer.render_preview(rt.RenderOptions(w, h, 1), gs, step, camera=rt_camera(rt, name))
    assert_same(got, full[ys][:, xs], "%s preview step %d" % (name, step))


def test_row_blocks_under_named_camera(rt, oracle, scenes):
    """rt_render_row_blocks with absolute rows: the ranks' stores into one device frame are the whole frame."""
    torch = pytest.importorskip("torch")
    from rtrace_b200 import partition
    gs, os_ = scenes
    w, h, spp = 200, 150, 2
    o = rt.RenderOptions(w, h, spp)
    for name in ("general", "mirrored"):
        ref, _ = os_.render(w, h, spp, camera=oracle_camera(oracle, name))
        for v in (rt.VARIANT_AUTO, rt.VARIANT_PHASED):
            frame = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
            rt.set_variant(v)
            try:
                for rank in range(3):
                    start, stride, blk, count = partition.block_band_spec(h, rank, 3, 16)
                    if count:
                        rt.Renderer.render_row_blocks(o, gs, start, stride, blk, count, frame.data_ptr(), pitch=w * 4,
                                                      absolute_rows=True, camera=rt_camera(rt, name),
                                                      stream=torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
            finally:
                rt.set_variant(rt.VARIANT_AUTO)
            assert_same(frame.cpu().numpy(), ref, "%s row blocks variant %d" % (name, v))


def test_sweeps_over_named_cameras(rt, oracle, scenes):
    """rt_render_sweep (RGBA and RGB) and rt_render_sweep_pull over every named camera."""
    gs, os_ = scenes
    w, h, spp = 192, 108, 2
    names = sorted(CAMS)
    refs = [os_.render(w, h, spp, camera=oracle_camera(oracle, n))[0] for n in names]
    cams = [rt_camera(rt, n) for n in names]
    o = rt.RenderOptions(w, h, spp)
    got, rgb = {}, {}
    rt.Renderer.render_sweep(o, gs, len(cams), cameras=cams, on_frame=lambda f, a: got.__setitem__(f, a.copy()))
    rt.Renderer.render_sweep(o, gs, len(cams), cameras=cams, rgb=True, on_frame=lambda f, a: rgb.__setitem__(f, a.copy()))
    assert sorted(got) == list(range(len(names))) and sorted(rgb) == sorted(got)
    for f, n in enumerate(names):
        assert_same(got[f], refs[f], "sweep frame %s" % n)
        assert_same(rgb[f], refs[f][:, :, :3], "RGB sweep frame %s" % n)
    base, _ = os_.render(w, h, spp)
    plan = [(100 + i, cams[i]) for i in range(len(cams))]
    plan.insert(3, (7, None))
    it = iter(plan)
    pulled = []
    rt.Renderer.render_sweep_pull(o, gs, lambda: next(it, None), on_frame=lambda f, a: pulled.append((f, a.copy())))
    assert [f for f, _ in pulled] == [p[0] for p in plan]
    for fid, img in pulled:
        assert_same(img, base if fid == 7 else refs[fid - 100], "pulled frame %d" % fid)


def test_multi_gpu_frame_under_named_camera(rt, oracle):
    if rt.device_count() < 2:
        pytest.skip("needs two GPUs")
    w, h, spp = 320, 180, 2
    scenes = []
    try:
        for g in range(2):
            rt.set_device(g)
            scenes.append(rt.Scene())
    finally:
        rt.set_device(0)
    for name in ("general", "sideways"):
        ref, _ = oracle.Scene().render(w, h, spp, camera=oracle_camera(oracle, name))
        assert_same(rt.Renderer.render_multi(rt.RenderOptions(w, h, spp), scenes, camera=rt_camera(rt, name)), ref, name)


def edge_camera(dev, seed):
    """A camera looking at the flake whose basis rows are off orthonormal by just under `dev` (f32 check)."""
    rot = _cameras.random_rotation(seed)
    b = _cameras.perturbed_basis(rot, dev, np.random.default_rng(seed))
    return (_cameras.CENTER - 4.2 * rot[2]).astype(F), b


def test_basis_just_inside_the_tolerance_runs_phased(rt, oracle, scenes):
    """A basis the host still accepts (rows within 1e-6 of orthonormal): a full 8K frame on PHASED equals the per-lane
    walk, and a small frame equals the oracle, on the fast variants."""
    gs, os_ = scenes
    tol = _cameras.host_tolerance()
    pair = edge_camera(0.97 * tol, 5)
    assert 0.8 * tol < _cameras.deviation32(pair[1]) <= tol and _cameras.orthonormal32(pair[1])
    cam = rt_camera(rt, pair)
    w, h, spp = 7680, 4320, 2
    o = rt.RenderOptions(w, h, spp)
    rt.set_variant(rt.VARIANT_PHASED)
    try:
        phased, st = rt.Renderer.render(o, gs, camera=cam, want_stats=True)
        assert st.variant_used == rt.VARIANT_PHASED
        rt.set_variant(rt.VARIANT_LANE)
        lane = rt.Renderer.render(o, gs, camera=cam)
    finally:
        rt.set_variant(rt.VARIANT_AUTO)
    assert (lane[:, :, 3] > 0).any()
    assert_same(phased, lane, "8K spp 2 PHASED vs LANE")
    del phased, lane
    w, h, spp = 320, 180, 2
    ref, okinds, _ = os_.render_region(w, h, spp, 0, 0, w, h, camera=oracle_camera(oracle, pair), kinds=True)
    for v in (rt.VARIANT_TILE, rt.VARIANT_PHASED):
        img, kinds, st = render_variant(rt, v, rt.RenderOptions(w, h, spp), gs, cam)
        assert st.variant_used == v
        assert np.array_equal(kinds, okinds)
        assert_same(img, ref, "inside the tolerance, variant %d" % v)


def test_basis_just_outside_the_tolerance_takes_the_lane_walk(rt, oracle, scenes):
    """Rows 1.5e-6 off orthonormal: outside what screen_box's slack is sized for, so every variant runs LANE and
    says so -- and returns the oracle's bytes."""
    gs, os_ = scenes
    tol = _cameras.host_tolerance()
    pair = edge_camera(1.5 * tol, 9)
    assert _cameras.deviation32(pair[1]) > 1.2 * tol and not _cameras.orthonormal32(pair[1])
    cam = rt_camera(rt, pair)
    w, h, spp = 320, 180, 2
    ref, okinds, _ = os_.render_region(w, h, spp, 0, 0, w, h, camera=oracle_camera(oracle, pair), kinds=True)
    for v in (rt.VARIANT_AUTO, rt.VARIANT_TILE, rt.VARIANT_PHASED):
        img, kinds, st = render_variant(rt, v, rt.RenderOptions(w, h, spp), gs, cam)
        assert st.variant_used == rt.VARIANT_LANE, (v, st.variant_used)
        assert np.array_equal(kinds, okinds)
        assert_same(img, ref, "outside the tolerance, variant %d" % v)


# ---- hand-built trees ---------------------------------------------------------------------------------------------

def flatten(node, sph, skip):
    """Pre-order flattening: node = (centre, radius) for a leaf, (centre, radius, [children]) for a group."""
    i = len(skip)
    sph.append(list(node[0]) + [node[1]])
    skip.append(0)
    for child in (node[2] if len(node) == 3 else ()):
        flatten(child, sph, skip)
    skip[i] = len(skip)
    return sph, skip


def rand_in_ball(rng, c, r):
    d = rng.normal(size=3)
    return np.asarray(c) + d / np.linalg.norm(d) * r * rng.random() ** (1 / 3)


def tree(kind, seed):
    rng = np.random.default_rng(seed)
    C0 = np.array([0.0, -1.0, 0.0])
    if kind == "overlapping_siblings":          # sibling bounds overlap each other heavily
        groups = []
        for _ in range(6):
            gc = rand_in_ball(rng, C0, 0.8)
            leaves = [(rand_in_ball(rng, gc, 0.6), rng.uniform(0.08, 0.3)) for _ in range(8)]
            groups.append((gc, 0.9, leaves))
        return (C0, 2.2, groups)
    if kind == "poking_out":                    # leaves reach past (or lie outside) their group's bound
        groups = []
        for _ in range(5):
            gc = rand_in_ball(rng, C0, 0.9)
            gr = rng.uniform(0.3, 0.6)
            leaves = [(gc + rng.normal(size=3) / 1.7 * gr * rng.uniform(0.5, 1.6), rng.uniform(0.1, 0.35))
                      for _ in range(7)]
            groups.append((gc, gr, leaves))
        return (C0, 1.6, groups)
    if kind == "duplicates":                    # the same sphere several times, in one group and across groups
        base = [(rand_in_ball(rng, C0, 1.0), rng.uniform(0.15, 0.4)) for _ in range(6)]
        g1 = (C0 + [0.2, 0, 0], 1.6, base[:4] + [base[1], base[2]])
        g2 = (C0 - [0.2, 0, 0], 1.6, [base[2], base[4], base[5], base[0]])
        return (C0, 2.0, [g1, base[3], g2, base[5]])
    if kind == "deep_chain":                    # one leaf and one nested group per level, 40 levels deep
        node = (C0 + [0.0, 0.0, -0.6], 0.2)
        for d in range(40):
            c = C0 + [0.9 * np.sin(d * 0.7), 0.6 * np.cos(d * 0.5), -0.6 + 0.03 * d]
            node = (c * 0.5 + C0 * 0.5, 0.25 + 0.05 * d, [(c, 0.06 + 0.004 * d), node])
        return (C0, 3.0, [node])
    if kind == "leaves_only":                   # the root holds leaves only
        return (C0, 2.0, [(rand_in_ball(rng, C0, 1.5), rng.uniform(0.03, 0.25)) for _ in range(300)])
    if kind == "eye_in_group":                  # the eye (0, 0, -4) lies inside a group bound in front of the flake
        near = (np.array([0.1, -0.3, -3.2]), 1.2,
                [(rand_in_ball(rng, [0.1, -0.3, -2.8], 0.5), rng.uniform(0.05, 0.15)) for _ in range(10)])
        far = (C0, 1.5, [(rand_in_ball(rng, C0, 1.1), rng.uniform(0.1, 0.3)) for _ in range(20)])
        return (np.array([0.0, -0.6, -1.8]), 3.5, [far, near])
    raise ValueError(kind)


LIGHT = tuple(_cameras.LIGHT)
TREES = [("overlapping_siblings", 1, LIGHT), ("poking_out", 2, LIGHT), ("duplicates", 3, tuple(_cameras.unit([0.4, -0.7, 0.6]))),
         ("deep_chain", 4, LIGHT), ("leaves_only", 5, tuple(_cameras.unit([-0.2, -0.5, -0.84]))),
         ("eye_in_group", 6, LIGHT), ("poking_out", 7, (-1.0, -3.0, 2.0))]   # the last light is not unit length


def tree_scenes(rt, oracle, kind, seed, light):
    sph, skip = flatten(tree(kind, seed), [], [])
    sph, skip = np.array(sph, F), np.array(skip, np.uint32)
    eye = (0.0, 0.0, -4.0)
    return rt.Scene.from_nodes(sph, skip, light, eye), oracle.Scene.from_nodes(sph, skip, light, eye), sph, skip


@pytest.mark.parametrize("kind,seed,light", TREES, ids=["%s-%d" % t[:2] for t in TREES])
def test_hand_built_tree_renders_match_oracle(rt, oracle, kind, seed, light):
    gs, os_, sph, skip = tree_scenes(rt, oracle, kind, seed, light)
    assert gs.counts() == os_.counts()
    assert np.array_equal(gs.light(), os_.light()) and np.array_equal(gs.light(), np.array(light, F))
    w, h, spp = 160, 120, 2
    for cam_name in (None, "roll30"):
        oc = None if cam_name is None else oracle_camera(oracle, cam_name)
        cam = None if cam_name is None else rt_camera(rt, cam_name)
        ref, okinds, ctr = os_.render_region(w, h, spp, 0, 0, w, h, camera=oc, kinds=True)
        assert ctr.primary_hits > 0
        for v in (rt.VARIANT_LANE, rt.VARIANT_WARP, rt.VARIANT_AUTO):
            img, kinds, st = render_variant(rt, v, rt.RenderOptions(w, h, spp), gs, cam)
            assert st.variant_used == (rt.VARIANT_WARP if v == rt.VARIANT_WARP else rt.VARIANT_LANE)
            assert np.array_equal(kinds, okinds), "%s camera %s: mask differs for variant %d" % (kind, cam_name, v)
            assert_same(img, ref, "%s camera %s variant %d" % (kind, cam_name, v))
        assert gs.count_rays(w, h, spp, camera=cam) == (ctr.primary_rays, ctr.shadow_rays)


@pytest.mark.parametrize("kind,seed,light", TREES[:6], ids=["%s-%d" % t[:2] for t in TREES[:6]])
def test_hand_built_tree_trace_rays_match_oracle(rt, oracle, kind, seed, light):
    gs, os_, sph, skip = tree_scenes(rt, oracle, kind, seed, light)
    rng = np.random.default_rng(seed + 100)
    n = 20000
    pos = rng.uniform([-3, -4, -5], [3, 2, 3], size=(n, 3)).astype(F)
    leaves = sph[skip == np.arange(1, len(skip) + 1)]
    aim = leaves[rng.integers(0, len(leaves), n), :3] + rng.normal(scale=0.2, size=(n, 3))
    dirs = np.where(rng.random((n, 1)) < 0.7, aim - pos, rng.normal(size=(n, 3)))
    dirs = (dirs / np.linalg.norm(dirs, axis=1, keepdims=True)).astype(F)
    gd, gn = gs.trace_rays(pos, dirs)
    od, on = os_.trace_rays(pos, dirs)
    hit = np.isfinite(od)
    assert hit.mean() > 0.3
    assert np.array_equal(gd, od), "%d of %d distances differ" % (int((gd != od).sum()), n)
    assert np.array_equal(gn[hit], on[hit])
