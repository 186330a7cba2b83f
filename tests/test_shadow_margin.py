"""PHASED decides whether a shadow ray is ever tested exactly with three bounds that are argued in comments of
rust-tracer_b200/csrc: K3 builds an origin segment and a scatter radius rho from a cull tile's hit range,
shadow_cover declares a whole tile occluded by one leaf, and the disc pre-filter (flush_shadow's radius R, K4's
projections) picks the candidates that get the exact any-hit test.  This CPU test restates them in numpy f32, one
rounding per operation (the library is built with -fmad=false; fmaf is one rounding), reads every constant they use
from the sources, and measures three claims:

1. every shadow origin K4 computes (render.rs:194-199) from a hit of the tile lies within rho of K3's segment;
2. a leaf shadow_cover accepts is hit by the exact f32 test from every point of that origin set: its true
   discriminant exceeds the worst-case f32 error EPS_DISC (v.v + r*r) (tests/test_cull_margin.py) everywhere;
3. the disc pre-filter, in K4's per-slot form (1 spp) and its packed FMA form (supersampled), keeps every
   (origin, candidate) pair whose exact test can pass.

The hits come from the oracle (oracle.trace_rays) for rays at the extreme sample positions of cull tiles of real
frames; synthetic leaves sit at the edge of each bound.  The approximate sqrt / division of the device (2 ulp) are
restated as correctly rounded ones: every bound here carries far more slack than that.  Each claim also asserts
that its smallest slack is small, so that the comparison measures something."""
import os
import re

import numpy as np
import pytest

import _cameras
from test_cull_margin import dot32, eps_disc, normalize32

F, D = np.float32, np.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rust-tracer_b200", "csrc")
PHASED = open(os.path.join(CSRC, "rt_phased.cu")).read()
CULL = open(os.path.join(CSRC, "rt_cull.cuh")).read()
NUM = r"([0-9.]+(?:e[+-]?[0-9]+)?)f"


def consts(src, pattern):
    """The numbers a source line is built from: the pattern (NUM marks each) must match exactly once."""
    m = re.findall(pattern.replace("NUM", NUM), src)
    assert len(m) == 1, "%r matches %d times: the restatement below no longer matches the source" % (pattern, len(m))
    return [F(v) for v in (m[0] if isinstance(m[0], tuple) else (m[0],))]


EPS = F(eps_disc())
# make_primary_beam (rt_cull.cuh)
HD_K, HD_C = consts(CULL, r"float hd = asqrt\(hx \* hx \+ hy \* hy\) \* NUM \+ NUM;")
CLEN_K, = consts(CULL, r"float clen = asqrt\(cx \* cx \+ cy \* cy \+ cz \* cz\) \* NUM;")
WIDE_K, = consts(CULL, r"pb\.wide = !\(clen > NUM \* hd\)")
TANP_K, TANP_C = consts(CULL, r"pb\.tanp = adiv\(hd, clen - hd\) \* NUM \+ NUM;")
SECP_K, = consts(CULL, r"pb\.secp = asqrt\(1\.0f \+ pb\.tanp \* pb\.tanp\) \* NUM;")
# K3's shadow beam (rt_phased.cu phase_cull_shadow)
OFF_K, OFF_C = consts(PHASED, r"const float off = thi \* NUM \+ NUM;")
A0_K, = consts(PHASED, r"float a0 = adiv\(tlo, pb\.secp\) \* NUM - off;")
RHO_T, RHO_K, RHO_C = consts(PHASED, r"sb\.rho = thi \* \(pb\.tanp \+ NUM\) \* NUM \+ NUM;")
RHO_WIDE_K, = consts(PHASED, r"sb\.rho = thi \* NUM \+ off;")
DEGEN_SIN, = consts(PHASED, r"sb\.degenerate = pb\.wide \|\| !\(sn > NUM\);")
# shadow_cover (rt_cull.cuh)
COV_DK, COV_DC = consts(CULL, r"const float D = fmaf\(asqrt\(fmaxf\(fmaxf\(d0, d1\), 0\.0f\)\), NUM, B\.rho \+ NUM\);")
COV_EK, COV_EC, COV_BK = consts(CULL, r"fmaf\(-D, D, rr\) >= NUM \* EPS_DISC \* fmaf\(vmax, vmax, rr\) \+ NUM && "
                                      r"bmin > NUM \* \(1\.0f \+ vmax\)")
# flush_shadow's disc radius (rt_phased.cu)
R_K, R_C = consts(PHASED, r"const float R = fmaf\(asqrt\(fmaf\(EPS_DISC, fmaf\(vmax, vmax, a\.w\), a\.w\)\), NUM, NUM\);")
SQRT_EPS = np.array([0x39b504f3], np.uint32).view(F)[0]   # K4: sqrt(f32::EPSILON) (render.rs:199)
assert "__uint_as_float(0x39b504f3u)" in PHASED

LIGHTS = {"default": (-1.0, -3.0, 2.0), "light_along_view": (0.0, 0.0, -1.0), "light_from_below": (0.3, 2.0, 0.5),
          "light_sideways": (-4.0, -0.2, 0.1)}   # test_gpu_parity.py test_other_scenes_match_oracle


def fma(a, b, c):
    """fmaf: the f32 product is exact in float64, so this rounds once more than the hardware only on ties."""
    return (np.asarray(a, D) * np.asarray(b, D) + np.asarray(c, D)).astype(F)


def lframe(light):
    """rt_api.cpp fill_params: e1, e2 perpendicular to the light, in float64, rounded to f32."""
    l = np.asarray(light, D) / np.linalg.norm(np.asarray(light, D))
    a = np.zeros(3)
    a[int(np.argmin(np.abs(l)))] = 1.0   # first axis least aligned with the light
    e1 = np.cross(l, a)
    e1 /= np.linalg.norm(e1)
    return e1.astype(F), np.cross(l, e1).astype(F)


class Frame:
    """A frame's camera and sampling: width x height (rows 0 ..), spp, eye and optional basis (rows right, up, fwd)."""

    def __init__(self, width, spp, eye, basis=None):
        self.w, self.h, self.spp = width, (width * 9) // 16, spp
        self.eye = np.asarray(eye, F)
        self.basis = None if basis is None else np.asarray(basis, F)
        self.bw, self.bh = (32, 16) if spp == 1 else (16, 8)   # PHASED's default cull tile
        self.frac = F(spp - 1) / F(spp)

    def dirs(self, x, y):
        """slot_dir (rt_cull.cuh, render.rs:238-243): unit f32 directions of sample positions x, y (f32 arrays)."""
        W, H = F(self.w), F(self.h)
        d = [x - W * F(0.5), (H - y) - H * F(0.5), np.full(x.shape, W, F)]
        if self.basis is not None:
            b = self.basis.reshape(9)
            d = [(b[k] * d[0] + b[3 + k] * d[1]) + b[6 + k] * d[2] for k in range(3)]
        return np.stack(normalize32(d), axis=1)

    def beam(self, ctx, cty):
        """cull_tile_beam + make_primary_beam: (axis, tanp, secp, wide) of cull tile (ctx, cty)."""
        x0, j0 = ctx * self.bw, cty * self.bh
        xh, jh = min(x0 + self.bw, self.w) - 1, min(j0 + self.bh, self.h) - 1
        x_lo, x_hi, y_lo, y_hi = F(x0), F(xh) + self.frac, F(j0), F(jh) + self.frac
        W, H = F(self.w), F(self.h)
        cx = F(0.5) * (x_lo + x_hi) - F(0.5) * W
        cy = (H - F(0.5) * (y_lo + y_hi)) - F(0.5) * H
        cz = W
        hx, hy = F(0.5) * (x_hi - x_lo), F(0.5) * (y_hi - y_lo)
        hd = np.sqrt(hx * hx + hy * hy) * HD_K + HD_C
        w = [cx, cy, cz]
        if self.basis is not None:
            b = self.basis.reshape(9)
            w = [(b[k] * cx + b[3 + k] * cy) + b[6 + k] * cz for k in range(3)]
        clen = np.sqrt((cx * cx + cy * cy) + cz * cz) * CLEN_K
        iw = F(1.0) / np.sqrt((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2])
        tanp = (hd / (clen - hd)) * TANP_K + TANP_C
        return (np.array([w[0] * iw, w[1] * iw, w[2] * iw], F), tanp, np.sqrt(F(1.0) + tanp * tanp) * SECP_K,
                not clen > WIDE_K * hd)

    def edge_samples(self, ctx, cty):
        """Sample positions on the border of the cull tile (every sub-sample step) and a coarse grid inside it."""
        step = F(1.0) / F(self.spp)
        x0, j0 = ctx * self.bw, cty * self.bh
        xs = F(x0) + step * np.arange((min(x0 + self.bw, self.w) - x0) * self.spp, dtype=F)
        ys = F(j0) + step * np.arange((min(j0 + self.bh, self.h) - j0) * self.spp, dtype=F)
        gx, gy = np.meshgrid(xs, ys)
        border = np.zeros(gx.shape, bool)
        border[[0, -1], :] = border[:, [0, -1]] = True
        border[::4, ::4] = True
        return gx[border].astype(F), gy[border].astype(F)


class ShadowBeam:
    """phase_cull_shadow: the origin segment P0 + s a, s in [0, len], and its scatter radius rho."""

    def __init__(self, eye, axis, tanp, secp, wide, tlo, thi, light):
        tlo, thi = F(tlo), F(thi)
        off = thi * OFF_K + OFF_C
        a0, a1 = (tlo / secp) * A0_K - off, thi + off
        if wide:
            a0 = a1 = F(0.0)
            self.rho = thi * RHO_WIDE_K + off
        else:
            self.rho = thi * (tanp + RHO_T) * RHO_K + RHO_C
        self.p0 = fma(a0, axis, eye)
        self.a = axis
        self.l = -np.asarray(light, F)   # render.rs:206
        self.len = a1 - a0
        n = np.cross(self.a.astype(D), self.l.astype(D))
        self.degenerate = wide or not np.linalg.norm(n) > DEGEN_SIN
        self.cosq = (self.a[0] * self.l[0] + self.a[1] * self.l[1]) + self.a[2] * self.l[2]

    def cover(self, c, r):
        """shadow_cover (rt_cull.cuh) for leaves c (n, 3) f32, radii r."""
        if self.degenerate:
            return np.zeros(len(r), bool)
        q = [c[:, k] - self.p0[k] for k in range(3)]
        qq = fma(q[0], q[0], fma(q[1], q[1], q[2] * q[2]))
        ql = fma(q[0], self.l[0], fma(q[1], self.l[1], q[2] * self.l[2]))
        qa = fma(q[0], self.a[0], fma(q[1], self.a[1], q[2] * self.a[2]))
        l1 = fma(-self.len, self.cosq, ql)
        d0 = fma(-ql, ql, qq)
        d1 = fma(-l1, l1, fma(self.len, self.len - F(2.0) * qa, qq))
        Dd = fma(np.sqrt(np.maximum(np.maximum(d0, d1), F(0.0))), COV_DK, self.rho + COV_DC)
        vmax = (np.sqrt(qq) + self.len) + self.rho
        rr = r * r
        bmin = np.minimum(ql, l1) - self.rho
        return (Dd < r) & (fma(-Dd, Dd, rr) >= (COV_EK * EPS) * fma(vmax, vmax, rr) + COV_EC) & \
            (bmin > COV_BK * (F(1.0) + vmax))

    def record(self, c, rr, e1, e2):
        """flush_shadow: the candidate's disc (cu, cv, R^2) in the plane perpendicular to the light."""
        q = [c[:, k] - self.p0[k] for k in range(3)]
        vmax = (np.sqrt(fma(q[0], q[0], fma(q[1], q[1], q[2] * q[2]))) + self.len) + self.rho
        R = fma(np.sqrt(fma(EPS, fma(vmax, vmax, rr), rr)), R_K, R_C)
        cu = fma(c[:, 0], e1[0], fma(c[:, 1], e1[1], c[:, 2] * e1[2]))
        cv = fma(c[:, 0], e2[0], fma(c[:, 1], e2[1], c[:, 2] * e2[2]))
        return cu, cv, R * R

    def worst(self, c, r):
        """float64: the smallest true discriminant and b = (c - o).L of the shadow rays from any origin of the set
        (within rho of the segment), and the largest |c - o|.  The distance from c to the shadow line through an
        origin is a norm of an affine function of the origin: largest at an end of the segment, plus rho."""
        q0 = c.astype(D) - self.p0.astype(D)
        q1 = q0 - D(self.len) * self.a.astype(D)
        L = self.l.astype(D) / np.linalg.norm(self.l.astype(D))
        perp = [np.linalg.norm(q - np.outer(q @ L, L), axis=1) for q in (q0, q1)]
        dmax = np.maximum(perp[0], perp[1]) + D(self.rho)
        vmax = np.maximum(np.linalg.norm(q0, axis=1), np.linalg.norm(q1, axis=1)) + D(self.rho)
        return r.astype(D) ** 2 - dmax ** 2, np.minimum(q0 @ L, q1 @ L) - D(self.rho), vmax

    def extreme_origins(self, c):
        """Per leaf: the ends of the segment pushed rho away from the leaf's shadow line (f32)."""
        L = self.l.astype(D) / np.linalg.norm(self.l.astype(D))
        out = []
        for end in (self.p0.astype(D), self.p0.astype(D) + D(self.len) * self.a.astype(D)):
            away = end - c.astype(D)
            away = away - np.outer(away @ L, L)
            away /= np.maximum(np.linalg.norm(away, axis=1), 1e-30)[:, None]
            out.append((end + D(self.rho) * away).astype(F))
        return out


def exact_hit(c, rr, o, to_light):
    """primitive.rs:56-68 as K4 restates it (shadow_test): finite distance <=> disc >= 0 and !(b + sqrt(disc) < 0)."""
    sv = [c[:, k] + (-o[:, k]) for k in range(3)]
    b = dot32(sv, to_light)
    disc = (b * b - dot32(sv, sv)) + rr
    with np.errstate(invalid="ignore"):
        return (disc >= F(0.0)) & ~(b + np.sqrt(np.maximum(disc, F(0.0))) < F(0.0))


def prefilter(o, cu, cv, R2, e1, e2, per_slot):
    """K4's disc test: per slot (1 spp) -- minus the origin's plane coordinates, then sums of squares -- or packed
    (supersampled): the same coordinates with FMAs and q = fma(dv, dv, du * du)."""
    no = [-o[:, 0], -o[:, 1], -o[:, 2]]
    nu = fma(no[0], e1[0], fma(no[1], e1[1], no[2] * e1[2]))
    nv = fma(no[0], e2[0], fma(no[1], e2[1], no[2] * e2[2]))
    du, dv = cu + nu, cv + nv
    q = (du * du + dv * dv) if per_slot else fma(dv, dv, du * du)
    return q <= R2, q


# ---------------------------------------------------------------------------------------------------------------
# real frames: cameras, widths, sample counts and scene levels
# ---------------------------------------------------------------------------------------------------------------
_SCENES = {}


def scene(level, light):
    import _oracle
    key = (level, light)
    if key not in _SCENES:
        s = _oracle.Scene(level=level, light=LIGHTS[light])
        sph, skip = s.flatten()
        leaf = skip == np.arange(1, len(skip) + 1)   # a leaf's skip pointer is the next node
        _SCENES[key] = (s, sph[leaf, :3].astype(F), sph[leaf, 3].astype(F), s.light())
    return _SCENES[key]


def frames():
    cams = [(None, None)] + [(None, _cameras.orbit_basis(f, 120)) for f in (7, 41)]
    named = _cameras.named_cameras()
    cams += [named[n] for n in ("general", "pitched_down", "off_light", "roll30")]
    out, i = [], 0
    for eye, basis in cams:
        for width in (1024, 3840, 65535):
            spp = 1 + (i * 3) % 8
            if eye is None and basis is not None:   # orbit camera: the reference eye (0, 0, -4) rotated, -4 forward
                eye = basis[2].astype(D) * -4.0
            out.append((Frame(width, spp, (0.0, 0.0, -4.0) if eye is None else eye, basis), 8 + i % 3,
                        list(LIGHTS)[i % 4]))
            i += 1
    return out


def tiles_with_hits(fr, os_, rng, n):
    """Up to n random cull tiles whose centre ray hits the scene: (ctx, cty, beam, origins, hit distances)."""
    ctx_n, cty_n = -(-fr.w // fr.bw), -(-fr.h // fr.bh)
    cand = rng.integers(0, ctx_n * cty_n, 40 * n)
    cx = (cand % ctx_n * fr.bw + fr.bw // 2).astype(F)
    cy = np.minimum(cand // ctx_n * fr.bh + fr.bh // 2, fr.h - 1).astype(F)
    dist, _ = os_.trace_rays(np.broadcast_to(fr.eye, (len(cand), 3)), fr.dirs(cx, cy))
    out = []
    for t in cand[np.isfinite(dist)][:n]:
        ctx, cty = int(t % ctx_n), int(t // ctx_n)
        x, y = fr.edge_samples(ctx, cty)
        d = fr.dirs(x, y)
        dist, nrm = os_.trace_rays(np.broadcast_to(fr.eye, (len(x), 3)), d)
        hit = np.isfinite(dist)
        d, dist, nrm = d[hit], dist[hit].astype(F), nrm[hit].astype(F)
        # render.rs:194-199 as K4 computes it: hit point eye + d t, then + normal * (t sqrt(eps))
        hp = fr.eye[None, :] + d * dist[:, None]
        o = hp + nrm * (dist * SQRT_EPS)[:, None]
        out.append((ctx, cty, fr.beam(ctx, cty), o.astype(F), dist))
    return out


@pytest.fixture(scope="module")
def real_tiles():
    rng = np.random.default_rng(20261020)
    out = []
    for fr, level, light in frames():
        os_, leaves, radii, lvec = scene(level, light)
        for ctx, cty, (axis, tanp, secp, wide), o, dist in tiles_with_hits(fr, os_, rng, 6):
            B = ShadowBeam(fr.eye, axis, tanp, secp, wide, dist.min(), dist.max(), lvec)
            out.append((fr, level, light, B, o))
    return out


def test_restated_frames_cover_the_ranges():
    """The frames span widths 1024 .. 65535, spp 1 .. 8, levels 8 .. 10 and the four lights."""
    fs = frames()
    assert {f.spp for f, _, _ in fs} == set(range(1, 9))
    assert {f.w for f, _, _ in fs} == {1024, 3840, 65535} and {lv for _, lv, _ in fs} == {8, 9, 10}
    assert {li for _, _, li in fs} == set(LIGHTS)


def test_shadow_origins_lie_within_rho_of_the_segment(real_tiles):
    """Claim 1: K4's shadow origins of a tile's hits are within rho of K3's segment built from their range."""
    worst = np.inf
    for fr, level, light, B, o in real_tiles:
        q = o.astype(D) - B.p0.astype(D)
        s = np.clip(q @ B.a.astype(D), 0.0, D(B.len))
        dist = np.linalg.norm(q - s[:, None] * B.a.astype(D)[None, :], axis=1)
        slack = (D(B.rho) - dist) / D(B.rho)
        assert slack.min() >= 0.0, "%dx%d spp %d: an origin lies %.3g past rho = %.3g" % (
            fr.w, fr.h, fr.spp, -slack.min() * B.rho, B.rho)
        worst = min(worst, float(slack.min()))
    assert len(real_tiles) >= 100
    assert np.isfinite(worst) and worst < 0.05, "smallest relative slack of rho: %g" % worst


def edge_leaves(B, rng, n, ks):
    """Synthetic leaves on the far side of the segment along the light, with radii such that their smallest true
    discriminant over the origin set is k EPS_DISC (vmax^2 + r^2) for each k in ks."""
    s = rng.uniform(0.0, 1.0, n) * D(B.len)
    t = rng.uniform(0.05, 3.0, n)
    L = B.l.astype(D) / np.linalg.norm(B.l.astype(D))
    side = np.cross(L, rng.normal(size=(n, 3)))
    side /= np.linalg.norm(side, axis=1)[:, None]
    c = B.p0.astype(D) + s[:, None] * B.a.astype(D) + t[:, None] * L + side * rng.uniform(0.0, 0.02, n)[:, None]
    c = c.astype(F)
    out_c, out_r = [], []
    for k in ks:
        r = np.full(n, 0.05)
        for _ in range(4):   # r^2 = dmax^2 + k EPS (vmax^2 + r^2): a fixed point, reached in a few steps
            disc, _, vmax = B.worst(c, r.astype(F))
            dmax2 = r ** 2 - disc
            r = np.sqrt(dmax2 + k * D(EPS) * (vmax ** 2 + r ** 2))
        out_c.append(c)
        out_r.append(r.astype(F))
    return np.concatenate(out_c), np.concatenate(out_r)


def test_shadow_cover_is_sound(real_tiles):
    """Claim 2: a leaf shadow_cover accepts -- scene leaves and synthetic leaves at the edge of its bound -- has a
    true discriminant above the worst-case f32 error and b > 0 from every origin of the set, and the exact f32 test
    hits it from the set's extreme points and from every real origin."""
    rng = np.random.default_rng(3)
    ks = np.geomspace(0.3, 6.0, 24)
    n_scene, tightest = 0, np.inf
    for fr, level, light, B, o in real_tiles:
        if B.degenerate:
            continue
        _, leaves, radii, lvec = scene(level, light)
        sc, sr = edge_leaves(B, rng, 8, ks)
        for c, r, synthetic in ((leaves, radii, False), (sc, sr, True)):
            acc = B.cover(c, r)
            if not acc.any():
                continue
            c, r = c[acc], r[acc]
            n_scene += 0 if synthetic else len(r)
            disc, bmin, vmax = B.worst(c, r)
            need = D(EPS) * (vmax ** 2 + r.astype(D) ** 2)
            assert (disc > need).all(), "%dx%d spp %d %s: an accepted leaf's discriminant is %.3g x the f32 error" % (
                fr.w, fr.h, fr.spp, light, float((disc / need).min()))
            assert (bmin > 4.0 * 2.0 ** -24 * vmax).all()
            tightest = min(tightest, float((disc / need).min()))
            to_light = [np.full(len(r), x, F) for x in B.l]
            for oe in B.extreme_origins(c):
                assert exact_hit(c, r * r, oe, to_light).all()
            for i in range(len(r)):
                tl = [np.full(len(o), x, F) for x in B.l]
                assert exact_hit(np.broadcast_to(c[i], o.shape), np.full(len(o), r[i] * r[i], F), o, tl).all()
    assert n_scene > 0, "no scene leaf covered a tile"
    assert np.isfinite(tightest) and tightest < 3.0 * COV_EK, "tightest accepted leaf: %.3g x the f32 error" % tightest


def test_disc_prefilter_keeps_every_pair_the_exact_test_accepts(real_tiles):
    """Claim 3 on real tiles: every (origin, scene leaf) pair whose exact f32 test hits passes K4's disc test with
    flush_shadow's radius, in the per-slot and the packed form."""
    worst, pairs = np.inf, 0
    for fr, level, light, B, o in real_tiles:
        _, leaves, radii, lvec = scene(level, light)
        e1, e2 = lframe(LIGHTS[light])
        L = B.l.astype(D)
        # leaves near the swept set (float64, generous): the exact test cannot reach the others
        q = leaves.astype(D) - B.p0.astype(D)
        near = np.linalg.norm(q - np.outer(q @ L, L), axis=1) < radii + D(B.len) + D(B.rho) + 0.01
        c, r = leaves[near], radii[near]
        if len(r) == 0:
            continue
        cu, cv, R2 = B.record(c, r * r, e1, e2)
        oi, ci = np.meshgrid(np.arange(len(o)), np.arange(len(r)), indexing="ij")
        oi, ci = oi.ravel(), ci.ravel()
        hit = exact_hit(c[ci], (r * r)[ci], o[oi], [np.full(len(oi), x, F) for x in B.l])
        if not hit.any():
            continue
        oi, ci = oi[hit], ci[hit]
        pairs += len(oi)
        for per_slot in (True, False):
            ok, qd = prefilter(o[oi], cu[ci], cv[ci], R2[ci], e1, e2, per_slot)
            assert ok.all(), "%dx%d spp %d %s: the disc test drops %d exact hits" % (fr.w, fr.h, fr.spp, light,
                                                                                     int((~ok).sum()))
            worst = min(worst, float(((R2[ci] - qd) / R2[ci]).min()))
    assert pairs > 1000
    assert np.isfinite(worst) and worst < 0.5, "smallest relative slack of R^2: %g" % worst


@pytest.mark.parametrize("light", list(LIGHTS))
def test_disc_prefilter_holds_at_the_edge_of_the_exact_test(light):
    """Claim 3 at its edge: synthetic pairs whose true distance from the candidate's centre to the shadow line is
    sqrt(r^2 + EPS_DISC (v.v + r^2)) -- the farthest the exact f32 test can accept -- with coordinates up to 15 and
    origin sets of one point (len = rho = 0, the tightest R), pass both forms of K4's disc test."""
    rng = np.random.default_rng(hash(light) % 2 ** 32)
    n = 200_000
    e1, e2 = lframe(LIGHTS[light])
    lv = np.asarray(LIGHTS[light], D)
    L = -(lv / np.linalg.norm(lv))
    o = rng.uniform(-15.0, 15.0, (n, 3)).astype(F)
    side = np.cross(L, rng.normal(size=(n, 3)))
    side /= np.linalg.norm(side, axis=1)[:, None]
    t = np.geomspace(0.01, 4.0, n)
    r = np.geomspace(1e-3, 0.5, n)[rng.permutation(n)]
    v2 = t ** 2   # |c - o|^2 to first order: refined below
    for _ in range(3):
        dist = np.sqrt(r ** 2 + D(EPS) * (v2 + r ** 2)) * (1.0 - 1e-7)
        v2 = t ** 2 + dist ** 2
    c = (o.astype(D) + t[:, None] * L + side * dist[:, None]).astype(F)
    keep = np.abs(c).max(axis=1) < 16.0
    o, c, r = o[keep], c[keep], r[keep].astype(F)
    worst = np.inf
    for k in range(len(o) // 20_000 + 1):
        sl = slice(k * 20_000, (k + 1) * 20_000)
        oo, cc, rr = o[sl], c[sl], r[sl]
        # flush_shadow with the origin set the single point o (P0 = o, len = rho = 0)
        qv = [cc[:, i] - oo[:, i] for i in range(3)]
        vmax = np.sqrt(fma(qv[0], qv[0], fma(qv[1], qv[1], qv[2] * qv[2])))
        R = fma(np.sqrt(fma(EPS, fma(vmax, vmax, rr * rr), rr * rr)), R_K, R_C)
        cu = fma(cc[:, 0], e1[0], fma(cc[:, 1], e1[1], cc[:, 2] * e1[2]))
        cv = fma(cc[:, 0], e2[0], fma(cc[:, 1], e2[1], cc[:, 2] * e2[2]))
        for per_slot in (True, False):
            ok, qd = prefilter(oo, cu, cv, R * R, e1, e2, per_slot)
            assert ok.all(), "%s: the disc test drops %d of %d pairs at the edge of the exact test" % (
                light, int((~ok).sum()), len(ok))
            worst = min(worst, float(((R * R - qd) / (R * R)).min()))
    assert np.isfinite(worst) and worst < 0.02, "smallest relative slack of R^2 at the edge: %g" % worst
