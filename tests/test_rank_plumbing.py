"""The one-process-per-GPU path against numpy and the oracle: what bench.py's band and frame records run under
torchrun (measure_bands, measure_frames) when every GPU has a process of its own.

A. rt_pack_rgb_rows (pack_rgb_blocks_kernel) against numpy on random RGBA: every width class, row-block layouts,
   partial last blocks, a height below the buffer's, the grid-stride loop, and the argument checks.
B. measure_bands' end-to-end plan run rank after rank in this process: render_row_blocks at absolute rows, pack,
   pitched copies into one page-locked /dev/shm frame; the frame must be the oracle's P6 body.
C. Two real processes (tests/_rank_worker.py): row blocks stored into another process's device frame through CUDA
   IPC, one shared host frame, and one shared frame queue.  The worker runs on device 1 as well when there is one.
"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _rank_worker as rw
from _rank_worker import SENTINEL

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = json.load(open(os.path.join(HERE, "golden", "oracle_derived.json")))

pytestmark = pytest.mark.gpu


def golden_case(width, height, spp, level):
    return next(c for c in GOLDEN["cases"] if (c["width"], c["height"], c["spp"], c["level"]) == (width, height, spp, level))


def p6_sha256(width, height, rgb):
    return hashlib.sha256(b"P6\n%d %d\n255\n" % (width, height) + rgb.tobytes()).hexdigest()


def oracle_camera(oracle, cam):
    oc = oracle.Camera()
    for k in ("eye", "right", "up", "forward"):
        getattr(oc, k)[:] = getattr(cam, k)[:]
    return oc


def shm_path(tag):
    return "/dev/shm/rtrace_test_%d_%s" % (os.getpid(), tag)


# ---- A. rt_pack_rgb_rows against numpy ---------------------------------------------------------------------------

WIDTHS = (1, 2, 3, 5, 7, 97, 1024, 7680, 65535)
LAYOUTS = ((1, 1), (4, 4), (16, 16), (32, 16), (48, 16), (128, 16), (64, 64))   # (row_stride, row_block)


def pack_cases():
    # only layouts whose blocks start at multiples of 4 pixels are accepted (test_pack_rejects_bad_arguments_...)
    cases = [(w, s, b) for w in WIDTHS for s, b in LAYOUTS if s * w % 4 == 0]
    # 524,280 quads a block, over the 1024 x 256 threads the launcher caps the grid at: each thread takes two
    cases.append((65535, 64, 32))
    return cases


def pack_plans(stride, block):
    """(row_start, height argument, buffer rows) triples for one layout."""
    part = block // 2 + 1 if block > 1 else 1        # rows of a partial last block: 3, 9, 33
    first1 = block if stride > block else stride     # the next rank's (or the next block's) first row
    plans = []
    for first in (0, first1):
        full = first + 2 * stride + block
        plans.append((first, full, full))                                # whole blocks, the gaps between them
        if block > 1:
            plans.append((first, first + stride + part, first + stride + part))   # partial last block
            plans.append((first, first + stride + part, full))           # ... and rows past `height` in the buffer
    plans.append((first1, first1, first1 + stride))                      # row_start >= height: nothing to do
    return plans


def expected_rgb(rgba, first, stride, block, height):
    exp = np.full(rgba.shape[:2] + (3,), SENTINEL, np.uint8)
    for y0 in range(first, height, stride):
        exp[y0:min(y0 + block, height)] = rgba[y0:min(y0 + block, height), :, :3]
    return exp


def download(rt, ptr, shape):
    out = np.empty(shape, np.uint8)
    rt.memcpy(out.ctypes.data, ptr, out.nbytes)
    return out


@pytest.mark.parametrize("width,stride,block", pack_cases(), ids=lambda v: str(v))
def test_pack_rgb_rows_matches_numpy(rt, width, stride, block):
    plans = pack_plans(stride, block)
    rows = max(p[2] for p in plans)
    rng = np.random.default_rng(width * 1000 + stride * 10 + block)
    rgba = rng.integers(0, 256, size=(rows, width, 4), dtype=np.uint8)   # alpha random too: a channel swap shows
    d_rgba, d_rgb = rt.device_alloc(rgba.nbytes), rt.device_alloc(rows * width * 3)
    try:
        rt.memcpy(d_rgba, rgba.ctypes.data, rgba.nbytes)
        for first, height, buf_rows in plans:
            rw.device_fill(d_rgb, buf_rows * width * 3)
            rt.pack_rgb_rows(d_rgba, d_rgb, width, height, first, stride, block)
            got = download(rt, d_rgb, (buf_rows, width, 3))
            exp = expected_rgb(rgba[:buf_rows], first, stride, block, height)
            if not np.array_equal(got, exp):
                bad = np.argwhere((got != exp).any(axis=-1))
                y, x = (int(v) for v in bad[0])
                raise AssertionError("width %d stride %d block %d row_start %d height %d (buffer %d rows): %d pixels "
                                     "differ, first at (row %d, col %d): got %s, expected %s"
                                     % (width, stride, block, first, height, buf_rows, len(bad), y, x,
                                        got[y, x].tolist(), exp[y, x].tolist()))
    finally:
        rt.device_free(d_rgba)
        rt.device_free(d_rgb)


def test_pack_rejects_bad_arguments_and_writes_nothing(rt):
    w, rows = 4, 65536   # sized so that even a launch over every row of every case stays inside the buffers
    n_rgba, n_rgb = w * rows * 4 + 64, w * rows * 3 + 64
    d_rgba, d_rgb = rt.device_alloc(n_rgba), rt.device_alloc(n_rgb)
    host_rgba, host_rgb = np.zeros(n_rgba, np.uint8), np.full(n_rgb, SENTINEL, np.uint8)
    other = None
    try:
        src = np.random.default_rng(1).integers(0, 256, n_rgba, dtype=np.uint8)
        rt.memcpy(d_rgba, src.ctypes.data, n_rgba)
        rw.device_fill(d_rgb, n_rgb)
        bad = [
            ("rgba 4 bytes off 16-byte alignment", (d_rgba + 4, d_rgb, w, 16, 0, 4, 4)),
            ("rgb 1 byte off 4-byte alignment", (d_rgba, d_rgb + 1, w, 16, 0, 4, 4)),
            ("row_start * width not a multiple of 4", (d_rgba, d_rgb, 5, 16, 1, 4, 4)),
            ("row_stride * width not a multiple of 4", (d_rgba, d_rgb, 5, 16, 0, 1, 1)),
            ("row_stride < row_block", (d_rgba, d_rgb, w, 16, 0, 4, 8)),
            ("row_block 0", (d_rgba, d_rgb, w, 16, 0, 4, 0)),
            ("NULL rgba", (0, d_rgb, w, 16, 0, 4, 4)),
            ("NULL rgb", (d_rgba, 0, w, 16, 0, 4, 4)),
            ("width 0", (d_rgba, d_rgb, 0, 16, 0, 4, 4)),
            ("height 0", (d_rgba, d_rgb, w, 0, 0, 4, 4)),
            ("width 65536", (d_rgba, d_rgb, 65536, 1, 0, 4, 4)),
            ("height 65536 at stride 1 (beyond the grid's y extent)", (d_rgba, d_rgb, w, 65536, 0, 1, 1)),
            ("host rgba", (host_rgba.ctypes.data, d_rgb, w, 16, 0, 4, 4)),
            ("host rgb", (d_rgba, host_rgb.ctypes.data, w, 16, 0, 4, 4)),
        ]
        if rt.device_count() >= 2:
            rt.set_device(1)
            try:
                other = rt.device_alloc(n_rgb)
            finally:
                rt.set_device(0)
            bad.append(("rgb on another device", (d_rgba, other, w, 16, 0, 4, 4)))
        for what, args in bad:
            with pytest.raises(rt.RtError) as e:
                rt.pack_rgb_rows(*args)
            assert e.value.code == rt.RT_ERR_INVALID, what
        assert (download(rt, d_rgb, (n_rgb,)) == SENTINEL).all()
        assert (host_rgb == SENTINEL).all()
        # the largest accepted frame height at stride 1 launches and packs
        rt.pack_rgb_rows(d_rgba, d_rgb, w, 65535, 0, 1, 1)
        rgba = download(rt, d_rgba, (n_rgba,))[:65535 * w * 4].reshape(65535, w, 4)
        assert np.array_equal(download(rt, d_rgb, (65535, w, 3)), rgba[..., :3])
    finally:
        rt.device_free(d_rgba)
        rt.device_free(d_rgb)
        if other is not None:
            rt.set_device(1)
            rt.device_free(other)
            rt.set_device(0)


# ---- B. measure_bands' end-to-end plan, rank after rank in this process ----------------------------------------

def band_e2e_frame(rt, width, height, spp, level, world, chunks, tag):
    """Every rank's packed blocks copied into one page-locked shared-memory frame; returns a copy of that frame."""
    path, nbytes = shm_path(tag), width * height * 3
    host = rw.SharedFile(path, nbytes, create=True)
    registered = False
    try:
        host.array[:] = SENTINEL
        rt.host_register(host.ptr, nbytes)
        registered = True
        rw.copy_out_ranks(rt.RenderOptions(width, height, spp), level, range(world), world, chunks, host.ptr)
        return host.array.reshape(height, width, 3).copy()
    finally:
        if registered:
            rt.host_unregister(host.ptr)
        host.close()
        os.unlink(path)


_oracle_frames = {}


def oracle_frame(oracle, width, height, spp, level):
    key = (width, height, spp, level)
    if key not in _oracle_frames:
        _oracle_frames[key] = oracle.Scene(level=level).render(width, height, spp)[0]
    return _oracle_frames[key]


@pytest.mark.parametrize("chunks", (1, 3))
@pytest.mark.parametrize("world", (1, 2, 3, 8))
@pytest.mark.parametrize("width,height,spp,level", ((97, 61, 2, 9), (200, 150, 4, 5)))
def test_band_e2e_plan_matches_oracle(rt, oracle, width, height, spp, level, world, chunks):
    frame = band_e2e_frame(rt, width, height, spp, level, world, chunks, "bands")
    ref = oracle_frame(oracle, width, height, spp, level)
    if not np.array_equal(frame, ref[..., :3]):
        bad = np.argwhere((frame != ref[..., :3]).any(axis=-1))
        raise AssertionError("%d pixels differ from the oracle, first at (row, col) %s" % (len(bad), tuple(bad[0])))
    assert p6_sha256(width, height, frame) == golden_case(width, height, spp, level)["ppm_sha256"]


def test_band_e2e_plan_c4_world8_matches_oracle_hash(rt):
    """bench's c4_bands record at N = 8 with its default 4 chunks: 7680x4320, 4x4 samples, level 9, a 99.5 MB
    shared frame."""
    width, height, spp, level = 7680, 4320, 4, 9
    frame = band_e2e_frame(rt, width, height, spp, level, 8, 4, "c4")
    assert p6_sha256(width, height, frame) == golden_case(width, height, spp, level)["ppm_sha256"]


# ---- C. two real processes ----------------------------------------------------------------------------------------

WORKER_DEVICES = pytest.mark.parametrize("worker_dev", (0, 1), ids=("same-device", "cross-device"))


def need_device(rt, dev):
    if dev >= rt.device_count():
        pytest.skip("needs %d CUDA devices" % (dev + 1))


class Worker:
    """tests/_rank_worker.py running `job` in a process of its own; killed and reaped on exit, whatever happens."""

    def __init__(self, job, timeout_s=180):
        env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "rust-tracer_b200"), HERE]))
        self.timeout_s = timeout_s
        self.proc = subprocess.Popen([sys.executable, os.path.join(HERE, "_rank_worker.py"), json.dumps(job)],
                                     env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)

    def alive(self):
        return self.proc.poll() is None

    def result(self):
        out, err = self.proc.communicate(timeout=self.timeout_s)
        assert self.proc.returncode == 0, "worker failed (exit %d):\n%s" % (self.proc.returncode, err[-4000:])
        return json.loads(out.strip().splitlines()[-1])

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        if self.proc.poll() is None:
            self.proc.kill()
        self.proc.wait()
        return False


SPLITS = pytest.mark.parametrize("world,worker_ranks", ((2, [1]), (3, [1])), ids=("world2", "world3"))


@SPLITS
@WORKER_DEVICES
def test_ipc_row_blocks_from_another_process(rt, oracle_scene8, worker_dev, world, worker_ranks):
    """The band kernel-only step: the worker's kernels store its row blocks straight into this process's device
    frame (rt_ipc_open); this process renders the other ranks' blocks into the same frame."""
    need_device(rt, worker_dev)
    width, height, spp, level = 200, 150, 2, 8
    opts = rt.RenderOptions(width, height, spp)
    nbytes = width * height * 4
    frame = rt.device_alloc(nbytes)
    try:
        rw.device_fill(frame, nbytes)
        job = dict(role="ipc_rows", device=worker_dev, handle=rt.ipc_export(frame).hex(), width=width, height=height,
                   spp=spp, level=level, world=world, ranks=worker_ranks)
        with Worker(job) as w:
            rw.render_ranks_into(opts, level, [r for r in range(world) if r not in worker_ranks], world, frame)
            assert w.result()["ok"]
        got = download(rt, frame, (height, width, 4))
    finally:
        rt.device_free(frame)
    ref, _ = oracle_scene8.render(width, height, spp)
    if not np.array_equal(got, ref):
        bad = np.argwhere((got != ref).any(axis=-1))
        raise AssertionError("%d pixels differ from the oracle, first at (row, col) %s" % (len(bad), tuple(bad[0])))


@SPLITS
@WORKER_DEVICES
def test_shared_host_frame_from_two_processes(rt, worker_dev, world, worker_ranks):
    """The band end-to-end step: both processes page-lock one shared-memory frame and copy their packed row blocks
    into it; the frame must be the oracle's P6 body."""
    need_device(rt, worker_dev)
    width, height, spp, level, chunks = 200, 150, 4, 5, 3
    path, nbytes = shm_path("host_frame"), width * height * 3
    host = rw.SharedFile(path, nbytes, create=True)
    registered = False
    try:
        host.array[:] = SENTINEL
        rt.host_register(host.ptr, nbytes)
        registered = True
        job = dict(role="host_frame", device=worker_dev, path=path, width=width, height=height, spp=spp, level=level,
                   world=world, chunks=chunks, ranks=worker_ranks)
        with Worker(job) as w:
            rw.copy_out_ranks(rt.RenderOptions(width, height, spp), level,
                              [r for r in range(world) if r not in worker_ranks], world, chunks, host.ptr)
            assert w.result()["ok"]
        frame = host.array.copy()
    finally:
        if registered:
            rt.host_unregister(host.ptr)
        host.close()
        os.unlink(path)
    assert p6_sha256(width, height, frame) == golden_case(width, height, spp, level)["ppm_sha256"]


@WORKER_DEVICES
def test_shared_frame_queue_across_processes(rt, oracle, oracle_scene8, worker_dev):
    """measure_frames' end-to-end sweep: both processes pull frame ids from one 64-bit counter in shared memory; every
    id is rendered exactly once, with its own orbit camera."""
    need_device(rt, worker_dev)
    width, height, spp, level, total = 160, 90, 2, 8, 16
    path = shm_path("queue")
    counter = rw.SharedFile(path, 64, create=True)
    try:
        job = dict(role="queue", device=worker_dev, path=path, width=width, height=height, spp=spp, level=level,
                   total=total, parties=2)
        with Worker(job) as w:
            scene = rt.Scene(level=level)
            mine = rw.pull_frames(rt.RenderOptions(width, height, spp), scene, counter.ptr, total, 2, alive=w.alive)
            scene.close()
            theirs = w.result()["frames"]
    finally:
        counter.close()
        os.unlink(path)
    ids = sorted(f for f, _ in mine + theirs)
    assert ids == list(range(total)), "ids %s" % ids
    for f, digest in mine + theirs:
        cam = rt.orbit_camera(rw.orbit_frame(f, total), rw.ORBIT_FRAMES)
        ref, _ = oracle_scene8.render(width, height, spp, camera=oracle_camera(oracle, cam))
        assert digest == hashlib.sha256(ref[..., :3].tobytes()).hexdigest(), "frame id %d" % f
