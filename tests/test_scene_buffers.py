"""The buffers a scene keeps between calls: the sweep's ring (regrown across output kinds, frame sizes and ring
depths), the per-stream scratch of the PHASED variant, and their release when the scene is closed.

Every frame a sweep delivers is compared byte for byte with the same scene's single-frame render of that camera
(for PNG and APNG, with the device encoder's file of that frame)."""
import contextlib
import os

import numpy as np
import pytest

N_FRAMES = 24  # the orbit the sweeps' cameras are taken from


@contextlib.contextmanager
def fresh_scene(rt):
    scene = rt.Scene()
    try:
        yield scene
    finally:
        scene.close()


def reference(rt, scene, kind, w, h, k, n):
    """What a `kind` sweep of n frames delivers for orbit frame k."""
    opts, cam = rt.RenderOptions(w, h, 1), rt.orbit_camera(k, N_FRAMES)
    if kind in ("rgba", "rgb"):
        img = rt.Renderer.render(opts, scene, camera=cam)
        return img if kind == "rgba" else np.ascontiguousarray(img[..., :3])
    ptr = rt.device_alloc(w * h * 4)
    try:
        rt.Renderer.render(opts, scene, camera=cam, out_ptr=ptr)
        return rt.encode_png(ptr, w, h) if kind == "png" else rt.encode_apng_frame(ptr, w, h, k, n)
    finally:
        rt.device_free(ptr)


def sweep(rt, scene, kind, w, h, n=4):
    """Runs a `kind` sweep of n orbit frames at w x h and checks every delivered frame."""
    opts, cams = rt.RenderOptions(w, h, 1), [rt.orbit_camera(k, N_FRAMES) for k in range(n)]
    got = {}

    def keep(f, frame):
        got[f] = frame if isinstance(frame, bytes) else frame.copy()

    if kind in ("rgba", "rgb"):
        rt.Renderer.render_sweep(opts, scene, n, cameras=cams, on_frame=keep, rgb=kind == "rgb")
    elif kind == "png":
        rt.Renderer.render_sweep_png(opts, [scene], n, cameras=cams, on_frame=keep)
    else:
        rt.Renderer.render_sweep_apng(opts, [scene], n, cameras=cams, on_frame=keep)
    assert sorted(got) == list(range(n)), (kind, w, h)
    for k in range(n):
        ref = reference(rt, scene, kind, w, h, k, n)
        if isinstance(ref, bytes):
            assert got[k] == ref, "%s %dx%d frame %d" % (kind, w, h, k)
        else:
            assert np.array_equal(got[k], ref), "%s %dx%d frame %d" % (kind, w, h, k)


REGROWTH = [("rgba", 160, 90), ("png", 1280, 720), ("rgb", 33, 7), ("apng", 640, 360), ("rgba", 1920, 1080)]


@pytest.mark.gpu
def test_sweep_ring_regrows_across_kinds_and_sizes(rt):
    with fresh_scene(rt) as scene:
        for kind, w, h in REGROWTH:
            sweep(rt, scene, kind, w, h)


@pytest.mark.gpu
def test_sweep_ring_depth_change(rt):
    """One render stream (two ring buffers), then the default two (three buffers), on the same scene."""
    saved = os.environ.pop("RTRACE_SWEEP_STREAMS", None)
    try:
        with fresh_scene(rt) as scene:
            os.environ["RTRACE_SWEEP_STREAMS"] = "1"
            for kind, w, h in REGROWTH[:3]:
                sweep(rt, scene, kind, w, h)
            del os.environ["RTRACE_SWEEP_STREAMS"]
            for kind, w, h in REGROWTH[:3]:
                sweep(rt, scene, kind, w, h)
    finally:
        os.environ.pop("RTRACE_SWEEP_STREAMS", None)
        if saved is not None:
            os.environ["RTRACE_SWEEP_STREAMS"] = saved


@pytest.mark.gpu
def test_phased_scratch_regrows(rt):
    """The PHASED scratch grows for a larger frame and is reused, not shrunk, for a smaller one."""
    with fresh_scene(rt) as scene:
        try:
            for w, h in ((512, 288), (2560, 1440), (512, 288)):
                opts = rt.RenderOptions(w, h, 1)
                rt.set_variant(rt.VARIANT_LANE)
                ref = rt.Renderer.render(opts, scene)
                rt.set_variant(rt.VARIANT_PHASED)
                img, st = rt.Renderer.render(opts, scene, want_stats=True)
                assert st.variant_used == rt.VARIANT_PHASED and st.kernel_launches == 4
                assert np.array_equal(img, ref), "%dx%d" % (w, h)
                assert len(rt.debug_phased_tiles(scene)) > 0
        finally:
            rt.set_variant(rt.VARIANT_AUTO)


@pytest.mark.gpu
def test_closed_scenes_return_their_device_memory(rt):
    """8 scenes, each holding a 4K sweep ring, PNG encoder scratch and PHASED scratch (a few hundred MB), are
    created and closed: free device memory comes back to within 64 MiB of where it was."""
    import torch

    w, h = 3840, 2160
    opts = rt.RenderOptions(w, h, 1)
    cams = [rt.orbit_camera(k, N_FRAMES) for k in range(3)]

    def use_and_close_a_scene():
        with fresh_scene(rt) as scene:
            rt.Renderer.render_sweep_png(opts, [scene], 3, cameras=cams)
            rt.set_variant(rt.VARIANT_PHASED)
            try:
                _, st = rt.Renderer.render(opts, scene, want_stats=True)
            finally:
                rt.set_variant(rt.VARIANT_AUTO)
            assert st.variant_used == rt.VARIANT_PHASED

    use_and_close_a_scene()  # loads the kernels this workload runs before the baseline is taken
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for _ in range(8):
        use_and_close_a_scene()
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    assert free0 - free1 <= 64 << 20, "%.1f MiB not returned" % ((free0 - free1) / 2**20)
