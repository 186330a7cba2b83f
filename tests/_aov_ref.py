"""Checks of AOV frames (include/rtrace.h "geometry output") against the pinned CPU oracle.  TEST INFRASTRUCTURE.

The AOV oracle (tests/_oracle_aov.cpp orc_render_rows_aov) has a sample loop of its own; these checks tie its output
to the pinned library (oracle/liboracle_rt.so) through two of its own entry points:
  * coverage: times spp*spp it is the number of samples that orc_render_region classifies as anything but
    background, so coverage == f32(count) * recip(spp*spp) bit for bit;
  * distance, normal, position: orc_trace_rays of every sample's primary ray (built as render_pixel builds it, with
    the camera extension) gives each sample's hit; the pixel's values follow in f32 from the contract's definition.
Used by tests/test_aov.py and tests/golden/make_aov_golden.py."""
import threading

import numpy as np

F = np.float32


def recip(spp):
    return F(1.0) / (F(spp) * F(spp))


def sample_dirs(w, h, spp, rows, basis=None):
    """Unit f32 directions of every sample of image rows `rows`, shape (len(rows), w, spp*spp, 3), samples in
    reference order (ssx outer, ssy inner; render.rs:236-243, oracle_rt.cpp render_pixel)."""
    ss = np.arange(spp, dtype=F) / F(spp)
    x = np.arange(w, dtype=F)[None, :, None, None] + ss[None, None, :, None]      # xres: ssx on axis 2
    y = np.asarray(rows, F)[:, None, None, None] + ss[None, None, None, :]        # yres: ssy on axis 3
    x, y = np.broadcast_arrays(x, y)
    W, H = F(w), F(h)
    d = [x - W / F(2.0), (H - y) - H / F(2.0), np.full(x.shape, W, F)]
    if basis is not None:   # rows right, up, forward
        b = np.asarray(basis, F).reshape(9)
        d = [(b[k] * d[0] + b[3 + k] * d[1]) + b[6 + k] * d[2] for k in range(3)]
    k = F(1.0) / np.sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2])
    return np.stack([d[0] * k, d[1] * k, d[2] * k], axis=-1).reshape(len(rows), w, spp * spp, 3)


def expected_from_hits(dist, nrm, eye, dirs, spp):
    """The AOV pixels from each sample's primary hit: dist (..., S) (+inf = miss), nrm and dirs (..., S, 3)."""
    S = dist.shape[-1]
    hit = dist != F(np.inf)
    n = np.zeros(dist.shape[:-1] + (3,), F)
    cnt = np.zeros(dist.shape[:-1], F)
    dmin = np.full(dist.shape[:-1], np.inf, F)
    pos = np.zeros(dist.shape[:-1] + (3,), F)
    eye = np.asarray(eye, F)
    for s in range(S):   # reference order: f32 sums in sample order, the first sample wins a tie
        h = hit[..., s]
        n = np.where(h[..., None], n + nrm[..., s, :], n)
        cnt = np.where(h, cnt + F(1.0), cnt)
        closer = h & (dist[..., s] < dmin)
        with np.errstate(invalid="ignore"):
            p = eye + dirs[..., s, :] * dist[..., s, None]
        dmin = np.where(closer, dist[..., s], dmin)
        pos = np.where(closer[..., None], p, pos)
    r = recip(spp)
    return np.concatenate([n * r, (cnt * r)[..., None], dmin[..., None], pos], axis=-1).astype(F)


def check_rows_against_traced_rays(aov_rows, pinned, w, h, spp, rows, eye, basis=None):
    """aov_rows (len(rows), w, 8) must be what orc_trace_rays' per-sample hits give, bit for bit."""
    dirs = sample_dirs(w, h, spp, rows, basis)
    pos = np.broadcast_to(np.asarray(eye, F), dirs.reshape(-1, 3).shape)
    dist, nrm = pinned.trace_rays(pos, dirs.reshape(-1, 3))
    want = expected_from_hits(dist.reshape(dirs.shape[:-1]), nrm.reshape(dirs.shape), eye, dirs, spp)
    assert_bits(aov_rows, want, "per-sample orc_trace_rays")


def covered_samples(pinned, w, h, spp, rows, camera=None, threads=8):
    """Per pixel of image rows `rows`: the number of samples orc_render_region does not classify as background.
    Runs of consecutive rows are rendered in parallel (ctypes releases the interpreter lock)."""
    rows = list(rows)
    out = np.empty((len(rows), w), np.int64)
    runs, start = [], 0
    for i in range(1, len(rows) + 1):
        if i == len(rows) or rows[i] != rows[i - 1] + 1:
            for a in range(start, i, 16):   # at most 16 rows per call
                runs.append((a, min(a + 16, i)))
            start = i
    lock = threading.Lock()

    def work():
        while True:
            with lock:
                if not runs:
                    return
                a, b = runs.pop()
            _, kinds, _ = pinned.render_region(w, h, spp, 0, rows[a], w, rows[b - 1] + 1, camera=camera, kinds=True)
            out[a:b] = (kinds != 0).sum(axis=-1)

    ts = [threading.Thread(target=work) for _ in range(threads)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return out


def check_rows_coverage(aov_rows, pinned, w, h, spp, rows, camera=None):
    """coverage == f32(covered samples) * recip(spp*spp), bit for bit."""
    cnt = covered_samples(pinned, w, h, spp, rows, camera)
    assert_bits(aov_rows[..., 3:4], (cnt.astype(F) * recip(spp))[..., None], "coverage against the kinds")


def assert_bits(got, ref, what=""):
    """Equal bit for bit (-0.0 != 0.0, NaN == NaN of the same payload)."""
    assert got.shape == ref.shape and got.dtype == np.float32 and ref.dtype == np.float32, (what, got.shape, ref.shape)
    g, r = got.view(np.uint32), ref.view(np.uint32)
    if not np.array_equal(g, r):
        bad = (g != r).reshape(g.shape[0], g.shape[1], -1).any(axis=-1)
        ys, xs = np.nonzero(bad)
        raise AssertionError("%s: %d of %d pixels differ, first at row %d col %d: got %r ref %r" % (
            what, len(ys), bad.size, ys[0], xs[0], got[ys[0], xs[0]], ref[ys[0], xs[0]]))
