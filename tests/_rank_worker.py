"""One rank of a one-process-per-GPU job, in a process of its own.  TEST INFRASTRUCTURE (not collected by pytest).

tests/test_rank_plumbing.py starts it as a second process next to the test's own, which plays the other ranks:

    python _rank_worker.py '<job as JSON>'

It imports rtrace_b200 and numpy only (no torch), so it starts fast, and prints one JSON line with its results.
Jobs ("role" selects one; every job names its CUDA "device"):
  ipc_rows    open rank 0's device frame from "handle" (hex of rt_ipc_export) and store "ranks"' row blocks into it
              with absolute row addressing (the band kernel-only step of bench.py's measure_bands)
  host_frame  register the POSIX shared-memory frame at "path" and copy "ranks"' packed RGB8 row blocks into it (the
              band end-to-end step of measure_bands)
  queue       pull orbit frames from the 64-bit counter at "path" with rt_render_sweep_pull, as measure_frames' end-to-end
              sweep does; reports [frame id, sha256 of the RGB8 frame] per frame

The helpers below are the same steps the test runs in its own process.
"""
import hashlib
import json
import mmap
import os
import sys
import time

import numpy as np

import rtrace_b200 as rt
from rtrace_b200 import partition

BLOCK = 16            # measure_bands' row block
SENTINEL = 0xA5       # fills every buffer before a step: a byte nobody wrote keeps it
ORBIT_FRAMES = 120


def orbit_frame(k, total):
    """bench.orbit_frame: the k-th of a job's `total` frames, spread evenly over the 120-frame orbit."""
    return (k * ORBIT_FRAMES // max(total, 1)) % ORBIT_FRAMES


class SharedFile:
    """A POSIX shared-memory file mapped into this process; `ptr` is its address."""

    def __init__(self, path, nbytes, create=False):
        import ctypes
        if create:
            with open(path, "wb") as f:
                f.truncate(nbytes)
        self.f = open(path, "r+b")
        self.mm = mmap.mmap(self.f.fileno(), nbytes)
        self.array = np.frombuffer(self.mm, dtype=np.uint8)
        self.ptr = ctypes.addressof(ctypes.c_char.from_buffer(self.mm))

    def close(self):
        self.array = None
        self.ptr = None
        try:
            self.mm.close()
        except BufferError:   # a view is still alive; the mapping goes with the process
            pass
        self.f.close()


def device_fill(ptr, nbytes, value=SENTINEL):
    """Fill device memory and wait until the bytes have landed: a copy from pageable memory may return before its
    transfer completes, and another process may store into the buffer next."""
    fill = np.full(nbytes, value, np.uint8)   # named: a temporary's .ctypes.data dangles before the call runs
    rt.memcpy(ptr, fill.ctypes.data, nbytes)
    sync_default_stream(ptr)


def sync_default_stream(dev_ptr):
    """Wait for the work queued on the legacy default stream: a device-to-host cudaMemcpy into pageable memory is
    ordered after it and returns only when it has completed."""
    b = np.empty(1, np.uint8)
    rt.memcpy(b.ctypes.data, dev_ptr, 1)


def band_groups(height, rank, world, chunks, block=BLOCK):
    """measure_bands' end-to-end plan for one rank: its blocks (partition.block_band_spec) in `chunks` groups of
    consecutive blocks, each (first image row, blocks, rows)."""
    row_start, row_stride, _, my_rows = partition.block_band_spec(height, rank, world, block)
    n_blocks = (my_rows + block - 1) // block
    chunks = max(1, min(chunks, n_blocks))
    groups = []
    for c in range(chunks):
        b0, b1 = c * n_blocks // chunks, (c + 1) * n_blocks // chunks
        if b1 > b0:
            first = row_start + b0 * row_stride
            rows = sum(min(block, height - (row_start + b * row_stride)) for b in range(b0, b1))
            groups.append((first, b1 - b0, rows))
    return groups


def copy_out_band(opts, scene, rank, world, chunks, own, own_rgb, host, block=BLOCK):
    """measure_bands' end-to-end step for one rank: per group, render its blocks at their image rows of the
    frame-shaped device buffer `own`, pack them to RGB8 in the frame-shaped `own_rgb` and copy them into the host
    frame at `host` (pitched copies, the image's partial last block on its own).  Everything is queued on the default
    stream, in that order."""
    width, height = opts.width, opts.height
    rgb_row = width * 3
    row_stride = world * block
    for first, nb, rows in band_groups(height, rank, world, chunks, block):
        rt.Renderer.render_row_blocks(opts, scene, first, row_stride, block, rows, own, pitch=width * 4,
                                      absolute_rows=True)
        last = first + (nb - 1) * row_stride
        rt.pack_rgb_rows(own, own_rgb, width, min(height, last + block), first, row_stride, block)
        whole = nb if last + block <= height else nb - 1
        off, pitch = first * rgb_row, row_stride * rgb_row
        if whole:
            rt.memcpy2d_async(host + off, pitch, own_rgb + off, pitch, block * rgb_row, whole)
        if whole < nb:   # the image's partial last block
            rt.memcpy2d_async(host + last * rgb_row, pitch, own_rgb + last * rgb_row, pitch, (height - last) * rgb_row, 1)


def copy_out_ranks(opts, level, ranks, world, chunks, host):
    """copy_out_band for each rank of `ranks` in turn, each with its own scene replica and its own sentinel-filled
    device buffers; returns when every copy has landed in the host frame."""
    width, height = opts.width, opts.height
    own, own_rgb = rt.device_alloc(height * width * 4), rt.device_alloc(height * width * 3)
    try:
        for rank in ranks:
            scene = rt.Scene(level=level)
            device_fill(own, height * width * 4)
            device_fill(own_rgb, height * width * 3)
            copy_out_band(opts, scene, rank, world, chunks, own, own_rgb, host)
            sync_default_stream(own_rgb)
            scene.close()
    finally:
        rt.device_free(own)
        rt.device_free(own_rgb)


def render_ranks_into(opts, level, ranks, world, frame, block=BLOCK):
    """measure_bands' kernel-only step: each rank's row blocks stored at their image rows of the whole device frame
    `frame` (possibly another process's, opened through rt_ipc_open)."""
    for rank in ranks:
        scene = rt.Scene(level=level)
        start, stride, blk, count = partition.block_band_spec(opts.height, rank, world, block)
        if count:   # want_stats: the call waits for its kernels
            rt.Renderer.render_row_blocks(opts, scene, start, stride, blk, count, frame, pitch=opts.width * 4,
                                          absolute_rows=True, want_stats=True)
        scene.close()


def wait_until(word_ptr, value, timeout_s=120.0, alive=lambda: True):
    """Spin until the 64-bit word at word_ptr reaches `value` (read with a fetch-and-add of 0)."""
    t_end = time.time() + timeout_s
    while rt.atomic_fetch_add_u64(word_ptr, 0) < value:
        if time.time() > t_end or not alive():
            raise TimeoutError("the other process never reached the barrier")
        time.sleep(0.001)


def pull_frames(opts, scene, counter, total, parties, alive=lambda: True):
    """measure_frames' end-to-end sweep: frame ids come from the counter at `counter` (word 0; word 1 is a start
    barrier of `parties` processes), camera orbit_frame(id, total); returns [[id, sha256 of the RGB8 frame], ...]."""
    rt.atomic_fetch_add_u64(counter + 8, 1)
    wait_until(counter + 8, parties, alive=alive)
    got = []

    def next_frame():
        i = rt.atomic_fetch_add_u64(counter, 1)
        if i >= total:
            return None
        return i, rt.orbit_camera(orbit_frame(i, total), ORBIT_FRAMES)

    def on_frame(f, arr):
        got.append([f, hashlib.sha256(arr.tobytes()).hexdigest()])
    rt.Renderer.render_sweep_pull(opts, scene, next_frame, on_frame=on_frame, rgb=True)
    return got


def main(job):
    rt.set_device(job["device"])
    opts = rt.RenderOptions(job["width"], job["height"], job["spp"])
    out = {}
    if job["role"] == "ipc_rows":
        frame = rt.ipc_open(bytes.fromhex(job["handle"]))
        try:
            render_ranks_into(opts, job["level"], job["ranks"], job["world"], frame)
        finally:
            rt.ipc_close(frame)
    elif job["role"] == "host_frame":
        host = SharedFile(job["path"], opts.width * opts.height * 3)
        rt.host_register(host.ptr, opts.width * opts.height * 3)
        try:
            copy_out_ranks(opts, job["level"], job["ranks"], job["world"], job["chunks"], host.ptr)
        finally:
            rt.host_unregister(host.ptr)
            host.close()
    elif job["role"] == "queue":
        counter = SharedFile(job["path"], 64)
        scene = rt.Scene(level=job["level"])
        try:
            out["frames"] = pull_frames(opts, scene, counter.ptr, job["total"], job["parties"])
        finally:
            scene.close()
            counter.close()
    else:
        raise ValueError("unknown role %r" % job["role"])
    out["ok"] = True
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main(json.loads(sys.argv[1]))
