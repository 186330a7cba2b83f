"""PHASED keeps a primary candidate for a lane only if the lane's samples overlap the candidate's image-space box
(screen_box in rust-tracer_b200/csrc/rt_phased.cu).  The box maps v = c - eye into camera coordinates with the basis
ROWS, q = B v, while a ray's world direction is B^T d: the two are inverse only for an exactly orthonormal B.  The
host sends every basis that orthonormal() in rt_api.cpp accepts to TILE / PHASED, so the box must hold for every
such basis, with the rows' dot products off the identity's by up to that tolerance.

This CPU test restates screen_box in f32 (numpy, one rounding per operation) and checks, for scene spheres of
levels 8-10 and seeded cameras whose bases sit at the tolerance, that the box contains the exact image-space extent
(float64) of the sphere inflated by the worst-case rounding of the discriminant, sqrt(r^2 + EPS_DISC (v.v + r^2)):
the set of rays whose exact f32 test can pass (tests/test_cull_margin.py).  A wider tolerance in orthonormal() than
the box's slack can absorb shows up here without a GPU."""
import numpy as np
import pytest

import _cameras
from test_cull_margin import eps_disc

F = np.float32
D = np.float64
WIDTHS = (3840, 7680, 15360, 65535)


def fma(a, b, c):
    """fmaf: the f32 product is exact in float64, so this rounds once more than the hardware only on ties."""
    return (D(1.0) * np.asarray(a, D) * np.asarray(b, D) + np.asarray(c, D)).astype(F)


def screen_box(basis, v, rr, width, height):
    """rt_phased.cu screen_box: {x_lo, x_hi, y_lo, y_hi} in sample coordinates (x_res, y_res), NaN where the sphere
    is not strictly in front (no bound).  v: (n, 3) f32, rr = r*r f32, basis rows right, up, forward (f32)."""
    b = np.asarray(basis, F).reshape(9)
    vx, vy, vz = v[:, 0], v[:, 1], v[:, 2]
    vv = (vx * vx + vy * vy) + vz * vz
    qx = fma(vx, b[0], fma(vy, b[1], vz * b[2]))
    qy = fma(vx, b[3], fma(vy, b[4], vz * b[5]))
    qz = fma(vx, b[6], fma(vy, b[7], vz * b[8]))
    R = fma(np.sqrt(fma(F(eps_disc()), vv + rr, rr)), F(1.001), F(1e-5))
    front = qz > F(1.01) * R
    A = fma(qz, qz, -R * R)
    k = F(width) / A
    cx, cy = qx * qz * k, qy * qz * k
    hx, hy = R * np.sqrt(fma(qx, qx, A)) * k, R * np.sqrt(fma(qy, qy, A)) * k
    sx = fma(hx, F(1.0005), fma(np.abs(cx), F(1e-5), F(0.05)))
    sy = fma(hy, F(1.0005), fma(np.abs(cy), F(1e-5), F(0.05)))
    hw, hh = F(0.5) * F(width), F(0.5) * F(height)
    box = np.stack([(cx - sx) + hw, (cx + sx) + hw, hh - (cy + sy), hh - (cy - sy)], axis=1).astype(D)
    box[~front] = np.nan
    return box


def exact_extent(basis, v, r, width, height):
    """Extremes, in sample coordinates, of the raw directions d = (X, Y, W) whose world direction B^T d passes within
    R = sqrt(r^2 + EPS_DISC (v.v + r^2)) of the centre: the conic d^T B (v v^T - (v.v - R^2) I) B^T d >= 0, float64."""
    B = np.asarray(basis, F).astype(D).reshape(3, 3)
    v = v.astype(D)
    r2 = r.astype(D) ** 2
    vv = np.einsum("ni,ni->n", v, v)
    R2 = r2 + eps_disc() * (vv + r2)
    q = v @ B.T                                     # B v per sphere
    Q = q[:, :, None] * q[:, None, :] - ((vv - R2)[:, None, None] * (B @ B.T)[None])
    Q = Q.reshape(-1, 9)
    q00, q01, q02, q11, q12, q22 = Q[:, 0], Q[:, 1], Q[:, 2], Q[:, 4], Q[:, 5], Q[:, 8]

    def roots(a, b, c):                             # a t^2 + 2 b t + c = 0
        disc = b * b - a * c
        assert (disc > 0).all()
        s = np.sqrt(disc)
        return np.minimum((-b - s) / a, (-b + s) / a), np.maximum((-b - s) / a, (-b + s) / a)

    # for u = X / W the sample row t = Y / W exists iff the quadratic in t has a real root; likewise with the axes swapped
    u0, u1 = roots(q01 * q01 - q00 * q11, q01 * q12 - q11 * q02, q12 * q12 - q11 * q22)
    t0, t1 = roots(q01 * q01 - q00 * q11, q01 * q02 - q00 * q12, q02 * q02 - q00 * q22)
    return np.stack([width * u0 + width / 2, width * u1 + width / 2, height / 2 - width * t1, height / 2 - width * t0], axis=1)


def excess(box, ext):
    """How far (pixels) the exact extent reaches past the box on its worst side; <= 0 when the box contains it."""
    return np.max(np.stack([box[:, 0] - ext[:, 0], ext[:, 1] - box[:, 1], box[:, 2] - ext[:, 2], ext[:, 3] - box[:, 3]]), axis=0)


_SPHERES = {}


def scene_spheres(level):
    if level not in _SPHERES:
        import _oracle
        _SPHERES[level] = _oracle.Scene(level=level).flatten()[0]
    return _SPHERES[level]


def worst_excess(rng, dev, n_cameras, n_spheres, widths=WIDTHS):
    """{width: the largest excess} over seeded cameras looking at the flake from 3.3 .. 6 units, bases perturbed
    to row dot deviations of `dev` (0: the rotation rounded to f32), and random scene spheres of levels 8 .. 10."""
    worst = {w: -np.inf for w in widths}
    for i in range(n_cameras):
        rot = _cameras.random_rotation(int(rng.integers(1 << 31)))
        basis = _cameras.perturbed_basis(rot, dev, rng) if dev else rot.astype(F)
        assert _cameras.deviation32(basis) <= max(dev, 2.4e-7)
        eye = (_cameras.CENTER - rng.uniform(3.3, 6.0) * rot[2]).astype(F)
        sph = scene_spheres(8 + i % 3)
        sph = sph[rng.integers(0, len(sph), n_spheres)]
        v = (sph[:, :3] - eye).astype(F)
        r = sph[:, 3]
        for w in widths:
            h = (w * 9) // 16
            box = screen_box(basis, v, r * r, w, h)
            keep = ~np.isnan(box[:, 0])
            e = excess(box[keep], exact_extent(basis, v[keep], r[keep], w, h))
            worst[w] = max(worst[w], float(e.max()))
    return worst


def test_orbit_and_named_bases_pass_the_host_check():
    """The cameras the suite renders on the fast path do pass orthonormal(): a rotation rounded to f32 is off by ~1e-7."""
    tol = _cameras.host_tolerance()
    for n in (120, 24):
        for k in range(n):
            assert _cameras.orthonormal32(_cameras.orbit_basis(k, n)), "orbit_camera(%d, %d)" % (k, n)
    for name, (eye, basis) in _cameras.named_cameras().items():
        assert _cameras.orthonormal32(basis), name
        assert _cameras.deviation32(basis) <= 1e-6 <= tol, name


def test_named_cameras_are_general():
    """The named cameras are what the GPU camera tests render: most of them have no small basis entry, so every term
    of the rotation rows carries weight; one of them is mirrored."""
    cams = _cameras.named_cameras()
    for name in _cameras.FULL_BASIS:
        assert np.abs(cams[name][1]).min() >= 0.05, name
    assert np.linalg.det(cams["mirrored"][1].astype(D)) < -0.99


def test_screen_box_check_is_live():
    """With bases rounded from exact rotations the box contains the extent with room to spare, yet the margin is a
    finite number of pixels (the comparison measures something)."""
    worst = worst_excess(np.random.default_rng(11), 0.0, 12, 3000)
    for w, e in worst.items():
        assert np.isfinite(e) and e < 0.0, (w, e)
        assert e > -1.0, (w, e)


@pytest.mark.parametrize("width", WIDTHS)
def test_screen_box_holds_at_the_host_tolerance(width):
    """Bases whose rows are off orthonormal by as much as orthonormal() accepts still get boxes that contain every ray
    that can pass the exact test -- at 4K, 8K, 16K-wide and 65535-wide frames."""
    tol = _cameras.host_tolerance()
    worst = worst_excess(np.random.default_rng(20261020), tol, 48, 4000, widths=(width,))[width]
    assert worst <= 0.0, "at tolerance %.1e a %d-wide frame's box misses the exact extent by %.3f px" % (tol, width, worst)
