"""Camera bases for the camera tests.  TEST INFRASTRUCTURE (no device needed).

A camera maps the raw direction d = (X, Y, W) of render.rs:240-242 to the world direction
right*X + up*Y + forward*W (rt_device.cuh primary_dir, oracle_rt.cpp render_pixel).  The orbit
camera is a rotation about y only, so four of its nine basis entries are 0 and one is 1; the
named cameras here are built in float64 and rounded to f32 once, so that most of them have no
zero entry and each row of the rotation is exercised by the tests that render them.
"""
import math
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32

CENTER = np.array([0.0, -1.0, 0.0])                          # Scene::default's flake (render.rs:145-166)
LIGHT = np.array([-1.0, -3.0, 2.0]) / math.sqrt(14.0)        # its light, normalised: the direction light travels


def host_tolerance():
    """The tolerance of orthonormal() in rt_api.cpp: a camera basis within it may run TILE / PHASED."""
    src = open(os.path.join(ROOT, "rust-tracer_b200", "csrc", "rt_api.cpp")).read()
    body = re.search(r"bool orthonormal\(const float b\[9\]\) \{(.*?)\n\}", src, re.S).group(1)
    return float(re.search(r"\)\s*>\s*([0-9.eE+-]+)f\)\s*return false", body).group(1))


def deviation32(basis):
    """max |row_i . row_j - delta_ij| of a 3x3 basis (rows right, up, forward) evaluated as orthonormal() in
    rt_api.cpp does: f32 operations, one rounding each, (x*x' + y*y') + z*z' (the library is built with
    -ffp-contract=off)."""
    b = np.asarray(basis, F).reshape(3, 3)
    worst = F(0.0)
    for i in range(3):
        for j in range(i, 3):
            d = (b[i, 0] * b[j, 0] + b[i, 1] * b[j, 1]) + b[i, 2] * b[j, 2]
            worst = max(worst, abs(d - (F(1.0) if i == j else F(0.0))))
    return float(worst)


def orthonormal32(basis, tol=None):
    """orthonormal() of rt_api.cpp restated: every row dot product within `tol` of the identity's."""
    tol = host_tolerance() if tol is None else tol
    return deviation32(basis) <= F(tol)


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v)


def look_at(eye, target, roll_deg=0.0, world_up=(0.0, 1.0, 0.0)):
    """Basis (rows right, up, forward) of a camera at `eye` looking at `target`, rolled about its forward axis.
    The reference camera (eye (0,0,-4) looking along +z) is right (1,0,0), up (0,1,0): right x up = forward."""
    f = unit(np.asarray(target, np.float64) - np.asarray(eye, np.float64))
    r = unit(np.cross(world_up, f))
    u = np.cross(f, r)
    a = math.radians(roll_deg)
    r, u = math.cos(a) * r + math.sin(a) * u, -math.sin(a) * r + math.cos(a) * u
    return np.array([r, u, f])


def random_rotation(seed):
    """A seeded rotation (rows right, up, forward; det +1) from the QR decomposition of a Gaussian matrix."""
    q, r = np.linalg.qr(np.random.default_rng(seed).normal(size=(3, 3)))
    q = q * np.sign(np.diag(r))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return q.T


def rotate_towards(a, b, deg):
    """Unit vector `deg` degrees from unit a in the plane of a and b, turned towards b."""
    p = unit(b - np.dot(a, b) * a)
    t = math.radians(deg)
    return math.cos(t) * a + math.sin(t) * p


def basis_facing(forward, roll_deg=0.0):
    f = unit(forward)
    return look_at(np.zeros(3), f, roll_deg)


def _named():
    cams = {}
    cams["pitched_down"] = (np.array([0.4, 3.0, -1.2]), look_at([0.4, 3.0, -1.2], CENTER))
    cams["from_below"] = (np.array([-0.5, -5.0, -1.5]), look_at([-0.5, -5.0, -1.5], CENTER))
    cams["roll30"] = (np.array([1.1, 0.9, -3.6]), look_at([1.1, 0.9, -3.6], CENTER, 30.0))
    cams["roll90"] = (np.array([-0.7, 0.4, -3.9]), look_at([-0.7, 0.4, -3.9], CENTER, 90.0))
    g = random_rotation(20261020)
    cams["general"] = (CENTER - 4.2 * g[2], g)
    m = random_rotation(21).copy()
    m[0] = -m[0]                                                 # right negated: det -1
    cams["mirrored"] = (CENTER - 4.0 * m[2], m)
    b = basis_facing(LIGHT, 20.0)                                # primary beams parallel to the shadow rays
    cams["along_light"] = (CENTER - 4.2 * b[2], b)
    off = rotate_towards(LIGHT, unit([1.0, 0.2, 0.3]), 2.9)      # |beam axis x light| ~ 0.05 at the image centre
    b = basis_facing(off, -35.0)
    cams["off_light"] = (CENTER - 4.2 * b[2], b)
    # just outside the root bound (radius 3) and looking past the flake: many spheres behind the image plane
    eye = CENTER + 3.15 * unit([0.3, 0.35, -1.0])
    toward = unit(CENTER - eye)
    side = unit(np.cross(toward, [0.0, 1.0, 0.0]))
    cams["sideways"] = (eye, basis_facing(math.cos(math.radians(62.0)) * toward + math.sin(math.radians(62.0)) * side, 12.0))
    return cams


# cameras whose nine basis entries all have magnitude >= 0.05 (checked by the tests)
FULL_BASIS = ("roll30", "general", "mirrored", "along_light", "off_light", "sideways")


def named_cameras():
    """name -> (eye, basis) rounded to f32: basis rows right, up, forward."""
    return {k: (e.astype(F), b.astype(F)) for k, (e, b) in _named().items()}


def orbit_basis(frame, n_frames):
    """orbit_camera(frame, n_frames) of rtrace_b200 restated (no library needed): rows right, up, forward in f32."""
    th = 2.0 * math.pi * frame / n_frames
    c, s = math.cos(th), math.sin(th)
    if frame % n_frames == 0:
        c, s = 1.0, 0.0
    return np.array([[c, 0.0, -s], [0.0, 1.0, 0.0], [s, 0.0, c]], F)


def perturbed_basis(rot, dev, rng):
    """rot (rows, orthonormal) times I + S, S symmetric with entries of magnitude ~dev/2 and random signs, scaled so
    that the f32 row dot products of the result (deviation32) deviate from the identity's by as close to `dev` as
    f32 rounding allows without exceeding it.  Rows of (I + S) rot have Gram matrix (I + S)^2 = I + 2 S + S^2."""
    sg = rng.choice([-1.0, 1.0], size=(3, 3))
    s0 = np.triu(sg) + np.triu(sg, 1).T
    lo, hi = 0.0, dev
    best = np.asarray(rot, F)
    for _ in range(40):                                          # bisection on the scale of S
        mid = 0.5 * (lo + hi)
        b = ((np.eye(3) + mid * s0) @ np.asarray(rot, np.float64)).astype(F)
        if deviation32(b) <= dev:
            lo, best = mid, b
        else:
            hi = mid
    return best
