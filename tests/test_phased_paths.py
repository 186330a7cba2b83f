"""The PHASED variant's rarely taken paths against the oracle.

The rest of the suite pins each variant's default path.  PHASED (rt_phased.cu) also has code that runs only on
large frames, under a forced tile shape, when the candidate pool runs out, when a tile's shadow list passes
RT_SHADOW_CAP, when one leaf occludes every shadow ray of a tile, or when the output buffer's alignment rules out
the paired store.  Most of it exists to skip exact tests, where a subtle error turns into wrong pixels.  Each
test here forces such a path, checks that it really ran (rt_stats.variant_used and rt_debug_phased_tiles), and
compares the bytes with the oracle -- or, for frames too large for the CPU, with the per-lane walk (LANE, itself
pinned to the oracle) plus oracle rows at the seams of the tile grids."""
import concurrent.futures
import functools
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import _cameras

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PHASED_SRC = open(os.path.join(ROOT, "rust-tracer_b200", "csrc", "rt_phased.cu")).read()
CAMS = _cameras.named_cameras()
WALK, COVERED = 0xffffffff, 0xfffffffd   # rt_debug_phased_tiles: per-lane walk / one leaf occludes every shadow ray

# PHASED's tile shapes (rt_launch_render_phased): (spp, RTRACE_TILE_SHAPE) -> (PXW, PXH, CW, CH); a shape a sample
# count does not list runs shape 0.
SHAPES = {(1, 0): (2, 2, 2, 2), (1, 1): (2, 2, 4, 4), (1, 2): (4, 2, 1, 2), (1, 3): (2, 1, 2, 4), (1, 4): (2, 1, 1, 2),
          (1, 5): (2, 2, 4, 2), (1, 6): (2, 2, 2, 4), (2, 1): (1, 1, 4, 4), (4, 1): (1, 1, 4, 4)}
# cull tiles above which K1 walks once for 2 x 2 of them (launch_phased)
K1C_SWITCH = int(re.search(r"if \(nc > (\d+)u\) \{\s*const Geo<SPP, PXW, PXH, CW \* 2, CH \* 2>", PHASED_SRC).group(1))


def phased_shape(spp, shape=0):
    t = SHAPES.get((spp, shape), (2, 2, 2, 2) if spp == 1 else (1, 1, 2, 2))
    assert "launch_phased<%d, %d, %d, %d, %d>" % ((spp,) + t) in PHASED_SRC, (spp, shape, t)
    return t


class Geo:
    """Geo<SPP, PXW, PXH, CW, CH> of rt_phased.cu: pixel tiles (one warp) and cull tiles of a frame of `rows` rows."""

    def __init__(self, width, rows, spp, shape=0):
        pxw, pxh, cw, ch = phased_shape(spp, shape)
        self.tw, self.th = 8 * pxw, 4 * pxh
        self.bw, self.bh = self.tw * cw, self.th * ch
        self.ptiles_x, self.ptiles_y = -(-width // self.tw), -(-rows // self.th)
        self.ctiles_x, self.ctiles_y = -(-self.ptiles_x // cw), -(-self.ptiles_y // ch)
        self.n_ctiles = self.ctiles_x * self.ctiles_y


def assert_same(gpu, ref, what=""):
    if not np.array_equal(gpu, ref):
        diff = np.abs(gpu.astype(np.int16) - ref.astype(np.int16))
        diff = diff.max(axis=-1) if diff.ndim == 3 else diff
        ys, xs = np.nonzero(diff)[:2]
        raise AssertionError("%s: %d of %d pixels differ (max %d), first at row %d col %d: gpu %s ref %s" % (
            what, len(ys), diff.size, diff.max(), ys[0], xs[0], gpu[ys[0], xs[0]], ref[ys[0], xs[0]]))


def cam_pair(rt, oracle, cam):
    """cam: None (the scene's camera), ("orbit", frame, eye) or a name of _cameras.named_cameras()."""
    if cam is None:
        return None, None
    if cam[0] == "orbit":
        g = rt.orbit_camera(cam[1], 120, eye=cam[2])
        return g, oracle.make_camera(g.eye[:], g.right[:], g.up[:], g.forward[:])
    eye, b = CAMS[cam]
    return rt.make_camera(eye, b[0], b[1], b[2]), oracle.make_camera(eye, b[0], b[1], b[2])


def oracle_region(os_, w, h, spp, camera=None):
    """The oracle's whole frame with its per-sample kinds and ray counts, rendered in row bands on every core."""
    n = os.cpu_count() or 1
    step = max(1, -(-h // (4 * n)))
    bands = [(b, min(h, b + step)) for b in range(0, h, step)]
    with concurrent.futures.ThreadPoolExecutor(n) as ex:
        parts = list(ex.map(lambda bt: os_.render_region(w, h, spp, 0, bt[0], w, bt[1], camera=camera, kinds=True), bands))
    return (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
            (sum(p[2].primary_rays for p in parts), sum(p[2].shadow_rays for p in parts)))


def render(rt, variant, o, scene, **kw):
    """render_rows under a forced variant; returns its results with rt_stats last."""
    rt.set_variant(variant)
    try:
        return rt.Renderer.render_rows(o, scene, want_stats=True, **kw)
    finally:
        rt.set_variant(rt.VARIANT_AUTO)


def check_oracle_rows(os_, img, w, h, spp, row_start, row_stride, rows, ocam, what):
    for j in rows:
        ref, _ = os_.render_rows(w, h, spp, row_start + j * row_stride, 1, 1, camera=ocam)
        assert_same(img[j:j + 1], ref, "%s local row %d" % (what, j))


def super_tile_spread(counts, geo):
    """Per cull tile: does its primary count equal that of the first tile of its 2 x 2 super-tile?"""
    c = counts[:geo.n_ctiles, 0].reshape(geo.ctiles_y, geo.ctiles_x)
    first = np.repeat(np.repeat(c[::2, ::2], 2, axis=0), 2, axis=1)[:geo.ctiles_y, :geo.ctiles_x]
    return c == first


# ---------------------------------------------------------------------------------------------------------------
# (a) K1's shared walk (K1C = 2) at partial super-tiles
# ---------------------------------------------------------------------------------------------------------------
# name: (width, height, spp, row_start, row_stride, camera).  Every frame above the switch has an odd number of
# cull tiles on both axes, so its last super-tile row and column are clipped.
SHARED_CULL = {
    "spp1_9605x8001": (9605, 8001, 1, 0, 1, None),
    **{"spp%d_4805x4001" % s: (4805, 4001, s, 0, 1, None) for s in range(2, 9)},
    "spp2_4805x4001_general": (4805, 4001, 2, 0, 1, "general"),
    "spp2_4805x3969_below": (4805, 3969, 2, 0, 1, None),
    "spp2_7688x9000_rows1of3": (7688, 9000, 2, 1, 3, None),
}


@pytest.mark.parametrize("name", list(SHARED_CULL))
def test_shared_primary_cull_at_partial_super_tiles(rt, oracle, oracle_scene8, name):
    w, h, spp, r0, rs, cam = SHARED_CULL[name]
    rows = (h - r0 + rs - 1) // rs
    geo = Geo(w, rows, spp)
    above = geo.n_ctiles > K1C_SWITCH
    if name.endswith("_below"):
        assert not above and geo.n_ctiles > K1C_SWITCH - 1000
    else:
        assert above and geo.ctiles_x % 2 == 1 and geo.ctiles_y % 2 == 1 and geo.ptiles_x % 2 == 1, name
    o = rt.RenderOptions(w, h, spp)
    gcam, ocam = cam_pair(rt, oracle, cam)
    gs = rt.Scene()   # its own scratch: the supersampled winners of these frames take up to ~10 GB
    try:
        img, st = render(rt, rt.VARIANT_PHASED, o, gs, row_start=r0, row_stride=rs, row_count=rows, camera=gcam)
        assert st.variant_used == rt.VARIANT_PHASED
        tiles = rt.debug_phased_tiles(gs)
        lane, st = render(rt, rt.VARIANT_LANE, o, gs, row_start=r0, row_stride=rs, row_count=rows, camera=gcam)
        assert st.variant_used == rt.VARIANT_LANE
    finally:
        gs.close()
    assert_same(img, lane, "%s PHASED vs LANE" % name)
    del lane
    assert len(tiles) >= geo.n_ctiles
    assert not (tiles[:geo.n_ctiles, 0] == WALK).any()   # the pool held every primary list: K2's list path ran
    same = super_tile_spread(tiles, geo)
    if above:   # one walk per super-tile: all (up to four) headers got its chain, the clipped ones included
        assert same.all(), "%s: %d tiles differ from their super-tile" % (name, int((~same).sum()))
    else:       # one walk per cull tile
        assert not same.all()
    seams = [0, 2015, 2016, 2047, 2048, (geo.ctiles_y - 1) * geo.bh, rows - 1]
    check_oracle_rows(oracle_scene8, img, w, h, spp, r0, rs, seams, ocam, name)


# ---------------------------------------------------------------------------------------------------------------
# (b) every tile shape, one process per RTRACE_TILE_SHAPE value
# ---------------------------------------------------------------------------------------------------------------
SIZES = ((203, 77), (1285, 723))      # clip the 64 x 32 and the 16 x 8 cull tiles on both axes
SHAPE_CAMS = (("orbit", 17, (0.0, 0.0, -4.0)), "general")
BIG = (4805, 4001)                    # shape 4 at spp 1: 301 x 501 cull tiles of 16 x 8 pixels, above the switch


def shape_cases(rt, shape):
    """(id, variant, spp, size, camera, kinds) of one process: forced PHASED at spp 1 (spp 2 and 4 too for the shapes
    they have), forced TILE at spp 1 .. 4 for its shapes 0 .. 2, and AUTO where it picks TILE (1285 x 723, 1 spp)."""
    runs = [(rt.VARIANT_PHASED, 1)]
    if shape <= 1:
        runs += [(rt.VARIANT_PHASED, 2), (rt.VARIANT_PHASED, 4)]
    if shape <= 2:
        runs += [(rt.VARIANT_TILE, s) for s in (1, 2, 3, 4)]
    out = []
    for variant, spp in runs:
        for size in SIZES:
            for ci, cam in enumerate(SHAPE_CAMS):
                for kinds in (False, True):
                    out.append(("v%d_spp%d_%dx%d_c%d_k%d" % (variant, spp, size[0], size[1], ci, kinds), variant, spp,
                                size, cam, kinds))
    out.append(("auto_tile", rt.VARIANT_AUTO, 1, SIZES[1], None, True))
    return out


@functools.lru_cache(maxsize=None)
def oracle_frame(level, w, h, spp, cam):
    import _oracle
    os_ = _oracle.Scene(level=level)
    ocam = None
    if cam is not None:
        if cam[0] == "orbit":
            import rtrace_b200 as rt
            g = rt.orbit_camera(cam[1], 120, eye=cam[2])
            ocam = _oracle.make_camera(g.eye[:], g.right[:], g.up[:], g.forward[:])
        else:
            eye, b = CAMS[cam]
            ocam = _oracle.make_camera(eye, b[0], b[1], b[2])
    return oracle_region(os_, w, h, spp, ocam)


@pytest.mark.parametrize("shape", range(7))
def test_every_tile_shape_matches_oracle(rt, oracle, oracle_scene8, tmp_path, shape):
    cases = []
    for cid, variant, spp, (w, h), cam, kinds in shape_cases(rt, shape):
        gcam = cam_pair(rt, oracle, cam)[0]
        camera = [list(gcam.eye), list(gcam.right), list(gcam.up), list(gcam.forward)] if gcam else None
        cases.append(dict(id=cid, variant=variant, width=w, height=h, spp=spp, camera=camera, kinds=kinds, tiles=False))
    if shape == 4:
        for cid, variant in (("big_phased", rt.VARIANT_PHASED), ("big_lane", rt.VARIANT_LANE)):
            cases.append(dict(id=cid, variant=variant, width=BIG[0], height=BIG[1], spp=1, camera=None, kinds=False,
                              tiles=variant == rt.VARIANT_PHASED))
    (tmp_path / "cases.json").write_text(json.dumps(cases))
    env = dict(os.environ, RTRACE_TILE_SHAPE=str(shape),
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "rust-tracer_b200"), HERE]))
    subprocess.run([sys.executable, os.path.join(HERE, "_shape_worker.py"), str(tmp_path / "cases.json"), str(tmp_path)],
                   env=env, check=True, timeout=900)
    used = json.loads((tmp_path / "variants.json").read_text())
    for cid, variant, spp, (w, h), cam, kinds in shape_cases(rt, shape):
        expect = rt.VARIANT_TILE if variant == rt.VARIANT_AUTO else variant
        assert used[cid] == expect, (cid, used[cid])
        ref, okinds, _ = oracle_frame(8, w, h, spp, cam)
        assert_same(np.load(tmp_path / (cid + "_img.npy")), ref, "shape %d %s" % (shape, cid))
        if kinds:
            assert np.array_equal(np.load(tmp_path / (cid + "_kinds.npy")), okinds), "shape %d %s: kinds" % (shape, cid)
    if shape == 4:
        assert used["big_phased"] == rt.VARIANT_PHASED and used["big_lane"] == rt.VARIANT_LANE
        geo = Geo(BIG[0], BIG[1], 1, 4)
        assert geo.n_ctiles > K1C_SWITCH and geo.ctiles_x % 2 == 1 and geo.ctiles_y % 2 == 1
        img = np.load(tmp_path / "big_phased_img.npy")
        assert_same(img, np.load(tmp_path / "big_lane_img.npy"), "shape 4 %dx%d PHASED vs LANE" % BIG)
        tiles = np.load(tmp_path / "big_phased_tiles.npy")
        assert not (tiles[:geo.n_ctiles, 0] == WALK).any() and super_tile_spread(tiles, geo).all()
        seams = [0, 2015, 2016, 2047, 2048, (geo.ctiles_y - 1) * geo.bh, BIG[1] - 1]
        check_oracle_rows(oracle_scene8, img, BIG[0], BIG[1], 1, 0, 1, seams, None, "shape 4 big")


# ---------------------------------------------------------------------------------------------------------------
# (c) the fallbacks at every sample count
# ---------------------------------------------------------------------------------------------------------------
POOL_LADDER = ("64", "1024", "4096", "16384", "65536")
POOL_FRAME = (192, 108)


def tile_states(tiles, n):
    """Counts of the three pool outcomes over the first n tiles: primary list overflowed (both columns read the
    per-lane walk: K3 hands such a tile to the walk too), primary list kept but shadow list overflowed, both kept."""
    p, s = tiles[:n, 0], tiles[:n, 1]
    return int((p == WALK).sum()), int(((p != WALK) & (s == WALK)).sum()), int(((p != WALK) & (s != WALK)).sum())


@pytest.mark.parametrize("spp", range(1, 9))
def test_pool_ladder_matches_oracle(rt, oracle, spp):
    w, h = POOL_FRAME
    ref, okinds, counts = oracle_frame(8, w, h, spp, None)
    n = Geo(w, h, spp).n_ctiles
    o = rt.RenderOptions(w, h, spp)
    gs = rt.Scene()
    states = {}
    rt.set_variant(rt.VARIANT_PHASED)
    try:
        for units in POOL_LADDER:
            os.environ["RTRACE_POOL_UNITS"] = units
            img, kinds, st = rt.Renderer.render_rows(o, gs, kinds=True, want_stats=True)
            assert st.variant_used == rt.VARIANT_PHASED
            states[units] = tile_states(rt.debug_phased_tiles(gs), n)
            assert_same(img, ref, "spp %d pool of %s units" % (spp, units))
            assert np.array_equal(kinds, okinds), "spp %d pool of %s units: kinds" % (spp, units)
            assert gs.count_rays(w, h, spp) == counts, "spp %d pool of %s units: ray counts" % (spp, units)
    finally:
        os.environ.pop("RTRACE_POOL_UNITS", None)
        rt.set_variant(rt.VARIANT_AUTO)
        gs.close()
    # which tiles overflow depends on the order in which warps reach the pool counter: some rung mixes all three
    assert any(all(k > 0 for k in s) for s in states.values()), "spp %d: no rung mixes the three states: %s" % (spp, states)
    assert states[POOL_LADDER[0]][0] > 0


@pytest.mark.parametrize("spp", range(2, 9))
def test_shadow_cap_hands_tiles_to_the_walk(rt, oracle, spp):
    """A level-10 tile with more than RT_SHADOW_CAP shadow candidates takes the any-hit walk (normal pool)."""
    w, h, level = 320, 180, 10
    ref, okinds, _ = oracle_frame(level, w, h, spp, None)
    gs = rt.Scene(level=level)
    try:
        img, kinds, st = render(rt, rt.VARIANT_PHASED, rt.RenderOptions(w, h, spp), gs, kinds=True)
        assert st.variant_used == rt.VARIANT_PHASED
        tiles = rt.debug_phased_tiles(gs)[:Geo(w, h, spp).n_ctiles]
    finally:
        gs.close()
    capped = (tiles[:, 0] != WALK) & (tiles[:, 1] == WALK)
    listed = tiles[:, 1][(tiles[:, 1] != WALK) & (tiles[:, 1] != COVERED)]
    assert capped.any(), "spp %d: no tile passed the shadow cap (largest list %d)" % (spp, int(listed.max(initial=0)))
    assert_same(img, ref, "spp %d level %d" % (spp, level))
    assert np.array_equal(kinds, okinds), "spp %d: kinds" % spp


COVER_EYE = (0.3, 0.6, -3.4)   # just outside the root bound: big leaves fill whole cull tiles


@pytest.mark.parametrize("spp", range(1, 9))
def test_covered_tiles_match_oracle(rt, oracle, spp):
    """Tiles whose shadow rays one leaf occludes (shadow_cover) are marked occluded without a test: the oracle's
    bytes and kinds, at every sample count, for one orbit camera and one other light too."""
    w, h = (640, 360) if spp <= 2 else (400, 225)
    kw, cam = dict(eye=COVER_EYE), None
    if spp == 3:
        cam = ("orbit", 9, COVER_EYE)
    if spp == 6:
        kw["light"] = (-2.0, -3.0, 1.0)
    gs, os_ = rt.Scene(**kw), oracle.Scene(**kw)
    gcam, ocam = cam_pair(rt, oracle, cam)
    try:
        img, kinds, st = render(rt, rt.VARIANT_PHASED, rt.RenderOptions(w, h, spp), gs, kinds=True, camera=gcam)
        assert st.variant_used == rt.VARIANT_PHASED
        tiles = rt.debug_phased_tiles(gs)[:Geo(w, h, spp).n_ctiles]
    finally:
        gs.close()
    assert (tiles[:, 1] == COVERED).any(), "spp %d: no COVERED tile" % spp
    ref, okinds, _ = oracle_region(os_, w, h, spp, ocam)
    assert_same(img, ref, "spp %d %s" % (spp, kw))
    assert np.array_equal(kinds, okinds), "spp %d: kinds" % spp


# ---------------------------------------------------------------------------------------------------------------
# (d) stores into device buffers of every alignment, checked against a canary
# ---------------------------------------------------------------------------------------------------------------
CANARY = 0xA5
STORE_VARIANTS = (("PHASED", 1), ("PHASED", 2), ("PHASED", 5), ("TILE", 1), ("LANE", 1))
STORE_H = 37


def canary_render(rt, fill_bytes, call):
    """Fill a device buffer with the canary, run call(device_ptr) -> rt_stats, and return (host copy, stats)."""
    ptr = rt.device_alloc(fill_bytes)
    try:
        host = np.full(fill_bytes, CANARY, np.uint8)
        rt.memcpy(ptr, host.ctypes.data, fill_bytes)
        st = call(ptr)
        rt.memcpy(host.ctypes.data, ptr, fill_bytes)
    finally:
        rt.device_free(ptr)
    return host, st


def check_window(buf, offset, pitch, w, rows_ref, what):
    """rows_ref: {buffer row -> oracle row}; those rows' pixels must equal the oracle, every other byte the canary."""
    written = np.zeros(buf.size, bool)
    for r, ref in rows_ref.items():
        at = offset + r * pitch
        got = buf[at:at + w * 4].reshape(1, w, 4)
        assert_same(got, ref.reshape(1, w, 4), "%s row %d" % (what, r))
        written[at:at + w * 4] = True
    stray = np.nonzero(buf[~written] != CANARY)[0]
    assert len(stray) == 0, "%s: %d bytes outside the written pixels changed, first at byte %d" % (
        what, len(stray), int(np.nonzero(~written)[0][stray[0]]))


@pytest.mark.parametrize("variant,spp", STORE_VARIANTS, ids=["%s-spp%d" % v for v in STORE_VARIANTS])
@pytest.mark.parametrize("offset", (0, 4))
@pytest.mark.parametrize("pitch8", (True, False), ids=("pitch8", "pitch4"))
@pytest.mark.parametrize("w", (97, 98))
def test_stores_into_device_windows(rt, oracle_scene8, gpu_scene8, variant, spp, offset, pitch8, w):
    """PHASED's spp-1 kernel stores pixel pairs with one 8-byte store when the pointer and the pitch allow it, else two
    4-byte stores guarded per pixel.  Every variant must write exactly the frame's pixels -- dense, interleaved and
    block-interleaved at absolute rows -- and leave the row padding and the rows it does not own untouched."""
    from rtrace_b200 import partition
    h = STORE_H
    pitch = -(-(w + 1) * 4 // 8) * 8 + (0 if pitch8 else 4)   # at least (w + 1) * 4: a pixel of padding per row
    assert (pitch % 8 == 0) == pitch8 and pitch >= (w + 1) * 4
    ref, _ = oracle_scene8.render(w, h, spp)
    o = rt.RenderOptions(w, h, spp)
    v = getattr(rt, "VARIANT_" + variant)
    what = "%s spp %d w %d pitch %d offset %d" % (variant, spp, w, pitch, offset)
    rows13 = list(range(1, h, 3))
    start, stride, blk, count = partition.block_band_spec(h, 1, 3, 8)
    owned = partition.block_band_rows(h, 1, 3, 8)
    layouts = (
        ("dense", h, {j: ref[j] for j in range(h)},
         lambda p: rt.Renderer.render_rows(o, gpu_scene8, out_ptr=p + offset, pitch=pitch, row_count=h, want_stats=True)[1]),
        ("rows 1 of 3", len(rows13), {j: ref[y] for j, y in enumerate(rows13)},
         lambda p: rt.Renderer.render_rows(o, gpu_scene8, row_start=1, row_stride=3, row_count=len(rows13),
                                           out_ptr=p + offset, pitch=pitch, want_stats=True)[1]),
        ("blocks at absolute rows", h, {y: ref[y] for y in owned},
         lambda p: rt.Renderer.render_row_blocks(o, gpu_scene8, start, stride, blk, count, p + offset, pitch=pitch,
                                                 absolute_rows=True, want_stats=True)),
    )
    assert 0 < len(owned) < h
    rt.set_variant(v)
    try:
        for name, n_rows, rows_ref, call in layouts:
            buf, st = canary_render(rt, offset + n_rows * pitch + 64, call)
            assert st.variant_used == v, (what, name, st.variant_used)
            check_window(buf, offset, pitch, w, rows_ref, "%s, %s" % (what, name))
    finally:
        rt.set_variant(rt.VARIANT_AUTO)
