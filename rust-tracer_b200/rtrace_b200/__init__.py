"""rtrace_b200 -- ctypes binding of librtrace_b200.so (include/rtrace.h).

A thin mirror of the reference crate's public surface (src/rust/lib.rs:8:
``Scene, Renderer, RenderOptions``) over the C ABI, used by the parity tests and
bench.py.  Nothing here computes pixels: every call goes through the CUDA library
and raises ``RtError`` when it fails (there is no CPU fallback).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
PKG_DIR = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("RTRACE_B200_LIB") or os.path.join(PKG_DIR, "librtrace_b200.so")  # env: kernel experiments

RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_NOMEM, RT_ERR_BUFFER = 0, -1, -2, -3, -4
VARIANT_AUTO, VARIANT_LANE, VARIANT_WARP, VARIANT_TILE, VARIANT_PHASED = 0, 1, 2, 3, 4

# every symbol include/rtrace.h declares (tests check the library exports all of them)
ABI_SYMBOLS = [
    "rt_last_error", "rt_version", "rt_device_count", "rt_set_device", "rt_set_variant",
    "rt_scene_create", "rt_scene_create_default", "rt_scene_create_from_nodes", "rt_scene_destroy",
    "rt_scene_counts", "rt_scene_export_nodes", "rt_flatten_pyramid_host", "rt_scene_light", "rt_scene_eye",
    "rt_scene_device", "rt_render_region", "rt_render_preview", "rt_render_rows", "rt_render_row_blocks", "rt_render_frame", "rt_render_sweep", "rt_render_sweep_rgb",
    "rt_render_frame_multi", "rt_render_sweep_multi", "rt_render_sweep_pull", "rt_atomic_fetch_add_u64",
    "rt_count_rays", "rt_trace_rays", "rt_measure_fp32_peak", "rt_microbench_fp32", "rt_selftest_math", "rt_debug_phased_tiles", "rt_host_alloc", "rt_host_free", "rt_host_register", "rt_host_unregister", "rt_microbench_d2h", "rt_device_alloc", "rt_device_free", "rt_ipc_export", "rt_ipc_open", "rt_ipc_close", "rt_memcpy", "rt_memcpy2d_async", "rt_pack_rgb_rows",
    "rt_png_bound", "rt_encode_png", "rt_render_sweep_png",
    "rt_apng_bound", "rt_encode_apng_frame", "rt_render_sweep_apng",
    "rt_render_rows_f32", "rt_render_frame_multi_f32",
]


class RtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("rtrace_b200 error %d: %s" % (code, msg))
        self.code = code


class Camera(C.Structure):
    _fields_ = [("eye", C.c_float * 3), ("right", C.c_float * 3), ("up", C.c_float * 3), ("forward", C.c_float * 3)]


class Stats(C.Structure):
    _fields_ = [("primary_rays", C.c_uint64), ("shadow_rays", C.c_uint64), ("kernel_ms", C.c_double),
                ("total_ms", C.c_double), ("kernel_launches", C.c_uint32), ("gpus", C.c_uint32),
                ("variant_used", C.c_uint32), ("reserved", C.c_uint32)]


FRAME_CALLBACK = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint8), C.c_size_t)
NEXT_FRAME_CALLBACK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(Camera), C.POINTER(C.c_int))

_lib = None


def lib():
    """Load the CUDA library; fail loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `make lib` (or __graft_entry__.build()); there is no fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    if os.environ.get("RTRACE_B200_LIB"):   # an experiment build may predate newer entry points: bind what it has
        class _Tolerant:
            def __init__(self, real):
                object.__setattr__(self, "_real", real)

            def __getattr__(self, name):
                try:
                    return getattr(self._real, name)
                except AttributeError:
                    return type("_Missing", (), {"argtypes": None, "restype": None})()
        real, L = L, _Tolerant(L)
    vp, u32, u16, f32p, u8p = C.c_void_p, C.c_uint32, C.c_uint16, C.POINTER(C.c_float), C.c_void_p
    u64p, u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
    L.rt_last_error.restype = C.c_char_p
    L.rt_version.restype = C.c_char_p
    L.rt_device_count.restype = C.c_int
    L.rt_set_variant.argtypes = [C.c_int]
    L.rt_set_device.argtypes = [C.c_int]
    L.rt_scene_create.argtypes = [u32, f32p, C.c_float, f32p, f32p, C.POINTER(vp)]
    L.rt_scene_create_default.argtypes = [C.POINTER(vp)]
    L.rt_scene_create_from_nodes.argtypes = [u32, f32p, u32p, f32p, f32p, C.POINTER(vp)]
    L.rt_scene_destroy.argtypes = [vp]
    L.rt_scene_destroy.restype = None
    L.rt_scene_counts.argtypes = [vp, u64p, u64p]
    L.rt_scene_export_nodes.argtypes = [vp, f32p, u32p, u32, u32p]
    L.rt_flatten_pyramid_host.argtypes = [u32, f32p, C.c_float, f32p, u32p, u32, u32p]
    L.rt_scene_light.argtypes = [vp, f32p]
    L.rt_scene_eye.argtypes = [vp, f32p]
    L.rt_scene_device.argtypes = [vp]
    L.rt_render_region.argtypes = [vp, u16, u16, u16, u16, u16, u16, u16, u8p, C.c_size_t]
    L.rt_render_rows.argtypes = [vp, C.POINTER(Camera), u32, u32, u32, u32, u32, u32, u8p, C.c_size_t, u8p, vp,
                                 C.POINTER(Stats)]
    L.rt_render_row_blocks.argtypes = [vp, C.POINTER(Camera), u32, u32, u32, u32, u32, u32, u32, u8p, C.c_size_t,
                                       C.c_int, vp, C.POINTER(Stats)]
    L.rt_render_frame.argtypes = [vp, C.POINTER(Camera), u32, u32, u32, u8p, C.c_size_t, C.POINTER(Stats)]
    L.rt_render_preview.argtypes = [vp, C.POINTER(Camera), u32, u32, u32, u8p, C.c_size_t, vp]
    L.rt_render_sweep.argtypes = [vp, C.POINTER(Camera), u32, u32, u32, u32, FRAME_CALLBACK, vp, C.POINTER(Stats)]
    L.rt_render_sweep_rgb.argtypes = L.rt_render_sweep.argtypes
    L.rt_render_frame_multi.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(Camera), u32, u32, u32, u8p, C.c_size_t,
                                        C.POINTER(Stats)]
    L.rt_render_sweep_multi.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(Camera), u32, u32, u32, u32, C.c_int,
                                        FRAME_CALLBACK, vp, C.POINTER(Stats)]
    L.rt_render_sweep_pull.argtypes = [vp, NEXT_FRAME_CALLBACK, vp, u32, u32, u32, C.c_int, FRAME_CALLBACK, vp, C.POINTER(Stats)]
    L.rt_atomic_fetch_add_u64.argtypes = [vp, C.c_uint64]
    L.rt_atomic_fetch_add_u64.restype = C.c_uint64
    L.rt_count_rays.argtypes = [vp, C.POINTER(Camera), u32, u32, u32, u32, u32, u32, u64p, u64p]
    L.rt_trace_rays.argtypes = [vp, C.c_size_t, vp, vp]
    L.rt_measure_fp32_peak.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.rt_microbench_fp32.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double)]
    L.rt_selftest_math.argtypes = [u32, u32, u64p]
    L.rt_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.rt_device_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.rt_device_free.argtypes = [vp]
    L.rt_device_free.restype = None
    L.rt_ipc_export.argtypes = [vp, C.c_char_p]
    L.rt_ipc_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.rt_ipc_close.argtypes = [vp]
    L.rt_memcpy.argtypes = [vp, vp, C.c_size_t]
    L.rt_pack_rgb_rows.argtypes = [vp, vp, u32, u32, u32, u32, u32, vp]
    L.rt_memcpy2d_async.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.c_size_t, C.c_size_t, vp]
    L.rt_host_free.argtypes = [vp]
    L.rt_host_free.restype = None
    L.rt_host_register.argtypes = [vp, C.c_size_t]
    L.rt_host_unregister.argtypes = [vp]
    L.rt_microbench_d2h.argtypes = [C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_double)]
    L.rt_png_bound.argtypes = [u32, u32, C.POINTER(C.c_size_t)]
    L.rt_encode_png.argtypes = [vp, u32, u32, C.c_size_t, vp, C.c_size_t, C.POINTER(C.c_size_t), vp]
    L.rt_render_sweep_png.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(Camera), u32, u32, u32, u32, FRAME_CALLBACK, vp,
                                      C.POINTER(Stats)]
    L.rt_apng_bound.argtypes = [u32, u32, u32, C.POINTER(C.c_size_t)]
    L.rt_encode_apng_frame.argtypes = [vp, u32, u32, C.c_size_t, u32, u32, u16, u16, vp, C.c_size_t,
                                       C.POINTER(C.c_size_t), vp]
    L.rt_render_sweep_apng.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(Camera), u32, u32, u32, u32, u16, u16,
                                       FRAME_CALLBACK, vp, C.POINTER(Stats)]
    L.rt_render_rows_f32.argtypes = [vp, C.POINTER(Camera), u32, u32, u32, u32, u32, u32, vp, C.c_size_t, vp,
                                     C.POINTER(Stats)]
    L.rt_render_frame_multi_f32.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(Camera), u32, u32, u32, vp, C.c_size_t,
                                            C.POINTER(Stats)]
    if os.environ.get("RTRACE_B200_LIB"):
        L = real
    _lib = L
    return L


def _check(rc):
    if rc != RT_OK:
        raise RtError(rc, lib().rt_last_error().decode("utf-8", "replace"))


def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def device_count():
    return int(lib().rt_device_count())


def version():
    return lib().rt_version().decode()


def set_device(d):
    _check(lib().rt_set_device(int(d)))


def set_variant(v):
    _check(lib().rt_set_variant(int(v)))


def make_camera(eye, right=(1, 0, 0), up=(0, 1, 0), forward=(0, 0, 1)):
    cam = Camera()
    cam.eye[:] = [float(x) for x in eye]
    cam.right[:] = [float(x) for x in right]
    cam.up[:] = [float(x) for x in up]
    cam.forward[:] = [float(x) for x in forward]
    return cam


def orbit_camera(frame, n_frames, eye=(0.0, 0.0, -4.0)):
    """Camera extension (SURVEY F6): the reference camera rotated about the flake's
    vertical axis by 2 pi frame / n_frames.  Frame 0 is the reference camera."""
    import math
    th = 2.0 * math.pi * frame / n_frames
    c, s = math.cos(th), math.sin(th)
    if frame % n_frames == 0:
        c, s = 1.0, 0.0

    def rot(v):
        return (c * v[0] + s * v[2], v[1], -s * v[0] + c * v[2])

    return make_camera(rot(eye), rot((1, 0, 0)), (0, 1, 0), rot((0, 0, 1)))


def flatten_pyramid_host(level, origin=(0.0, -1.0, 0.0), radius=1.0):
    """Host-only scene flattening (no GPU needed)."""
    n = C.c_uint32()
    _check(lib().rt_flatten_pyramid_host(level, _f3(origin), radius, None, None, 0, C.byref(n)))
    sph = np.empty((n.value, 4), np.float32)
    sk = np.empty(n.value, np.uint32)
    _check(lib().rt_flatten_pyramid_host(level, _f3(origin), radius, _fp(sph), sk.ctypes.data_as(C.POINTER(C.c_uint32)),
                                         n.value, C.byref(n)))
    return sph, sk


class RenderOptions:
    """render.rs:33-38"""

    def __init__(self, width=1024, height=1024, samples_per_pixel=1):
        self.width, self.height, self.samples_per_pixel = int(width), int(height), int(samples_per_pixel)


class Scene:
    """render.rs:138-167 ``Scene``; ``Scene()`` is ``Scene::default()``."""

    def __init__(self, level=8, origin=(0.0, -1.0, 0.0), radius=1.0, light=(-1.0, -3.0, 2.0), eye=(0.0, 0.0, -4.0),
                 _handle=None):
        self._h = C.c_void_p()
        if _handle is not None:
            self._h = _handle
        else:
            _check(lib().rt_scene_create(level, _f3(origin), radius, _f3(light), _f3(eye), C.byref(self._h)))

    @classmethod
    def from_nodes(cls, spheres4, skip, light, eye):
        sph = np.ascontiguousarray(spheres4, dtype=np.float32)
        sk = np.ascontiguousarray(skip, dtype=np.uint32)
        h = C.c_void_p()
        _check(lib().rt_scene_create_from_nodes(len(sk), _fp(sph), sk.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                _f3(light), _f3(eye), C.byref(h)))
        return cls(_handle=h)

    def close(self):
        if getattr(self, "_h", None):
            lib().rt_scene_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def counts(self):
        g, i = C.c_uint64(), C.c_uint64()
        _check(lib().rt_scene_counts(self._h, C.byref(g), C.byref(i)))
        return g.value, i.value

    def export_nodes(self):
        n = C.c_uint32()
        _check(lib().rt_scene_export_nodes(self._h, None, None, 0, C.byref(n)))
        sph = np.empty((n.value, 4), np.float32)
        sk = np.empty(n.value, np.uint32)
        _check(lib().rt_scene_export_nodes(self._h, _fp(sph), sk.ctypes.data_as(C.POINTER(C.c_uint32)), n.value,
                                           C.byref(n)))
        return sph, sk

    def light(self):
        v = (C.c_float * 3)()
        _check(lib().rt_scene_light(self._h, v))
        return np.array(v[:], np.float32)

    def eye(self):
        v = (C.c_float * 3)()
        _check(lib().rt_scene_eye(self._h, v))
        return np.array(v[:], np.float32)

    def device(self):
        return int(lib().rt_scene_device(self._h))

    def trace_rays(self, pos, dirs):
        pos = np.asarray(pos, np.float32).reshape(-1, 3)
        dirs = np.asarray(dirs, np.float32).reshape(-1, 3)
        rays = np.ascontiguousarray(np.concatenate([pos, dirs], axis=1), np.float32)
        hits = np.empty((len(pos), 4), np.float32)
        _check(lib().rt_trace_rays(self._h, len(pos), rays.ctypes.data, hits.ctypes.data))
        return hits[:, 0].copy(), hits[:, 1:].copy()

    def count_rays(self, width, height, spp, row_start=0, row_stride=1, row_count=None, camera=None):
        row_count = height if row_count is None else row_count
        p, s = C.c_uint64(), C.c_uint64()
        _check(lib().rt_count_rays(self._h, C.byref(camera) if camera is not None else None, width, height, spp,
                                   row_start, row_stride, row_count, C.byref(p), C.byref(s)))
        return p.value, s.value


class Renderer:
    """render.rs:169-311 ``Renderer`` (associated functions only, like the reference)."""

    @staticmethod
    def render_region(options, scene, l, b, r, t):
        """Renderer::render_region (render.rs:218-255) -> (t-b, r-l, 4) uint8."""
        out = np.empty((max(t - b, 0), max(r - l, 0), 4), np.uint8)
        _check(lib().rt_render_region(scene.handle, options.width, options.height, options.samples_per_pixel,
                                      l, b, r, t, out.ctypes.data, out.nbytes))
        return out

    @staticmethod
    def render_rows(options, scene, row_start=0, row_stride=1, row_count=None, camera=None, kinds=False, out=None,
                    out_ptr=None, pitch=0, stream=None, want_stats=False):
        """One GPU's interleaved share of Renderer::render's bucket loop (render.rs:268-309)."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        if row_count is None:
            row_count = (h - row_start + row_stride - 1) // row_stride
        kd = None
        if out_ptr is None:
            if out is None:
                out = np.empty((row_count, w, 4), np.uint8)
            out_ptr = out.ctypes.data
        if kinds:
            kd = np.empty((row_count, w, spp * spp), np.uint8)
        st = Stats() if want_stats else None
        _check(lib().rt_render_rows(scene.handle, C.byref(camera) if camera is not None else None, w, h, spp,
                                    row_start, row_stride, row_count, out_ptr, pitch,
                                    kd.ctypes.data if kd is not None else None, stream,
                                    C.byref(st) if st is not None else None))
        res = [out]
        if kinds:
            res.append(kd)
        if want_stats:
            res.append(st)
        return res[0] if len(res) == 1 else tuple(res)

    @staticmethod
    def render_row_blocks(options, scene, row_start, row_stride, row_block, row_count, out_ptr, pitch=0,
                          absolute_rows=False, camera=None, stream=None, want_stats=False):
        """Rows in blocks of `row_block` consecutive image rows, `row_stride` apart (device output only)."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        st = Stats() if want_stats else None
        _check(lib().rt_render_row_blocks(scene.handle, C.byref(camera) if camera is not None else None, w, h, spp,
                                          row_start, row_stride, row_block, row_count, out_ptr, pitch,
                                          1 if absolute_rows else 0, stream, C.byref(st) if st is not None else None))
        return st

    @staticmethod
    def render(options, scene, camera=None, out=None, out_ptr=None, want_stats=False):
        """Renderer::render (render.rs:260-310): the whole frame on the scene's GPU."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        if out_ptr is None:
            if out is None:
                out = np.empty((h, w, 4), np.uint8)
            out_ptr = out.ctypes.data
        st = Stats() if want_stats else None
        _check(lib().rt_render_frame(scene.handle, C.byref(camera) if camera is not None else None, w, h, spp,
                                     out_ptr, w * h * 4, C.byref(st) if st is not None else None))
        return (out, st) if want_stats else out

    @staticmethod
    def render_f32(options, scene_or_scenes, camera=None, out_ptr=None, want_stats=False):
        """The frame before quantisation (rt_render_frame_multi_f32): (h, w, 4) float32 {r, g, b, alpha}, equal bit
        for bit to the reference's values.  A list of scenes renders on their GPUs; with out_ptr (device memory of
        the first scene's GPU, h * w * 16 bytes) the frame is stored there and None is returned in its place."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        scenes = list(scene_or_scenes) if isinstance(scene_or_scenes, (list, tuple)) else [scene_or_scenes]
        out = None
        if out_ptr is None:
            out = np.empty((h, w, 4), np.float32)
            out_ptr = out.ctypes.data
        arr = (C.c_void_p * len(scenes))(*[s.handle for s in scenes])
        st = Stats() if want_stats else None
        _check(lib().rt_render_frame_multi_f32(arr, len(scenes), C.byref(camera) if camera is not None else None, w, h,
                                               spp, out_ptr, w * h * 16, C.byref(st) if st is not None else None))
        return (out, st) if want_stats else out

    @staticmethod
    def render_rows_f32(options, scene, row_start=0, row_stride=1, row_count=None, camera=None, out=None,
                        out_ptr=None, pitch=0, stream=None, want_stats=False):
        """render_rows before quantisation (rt_render_rows_f32): (row_count, w, 4) float32 for host output; with
        out_ptr (host or device memory, `pitch` bytes per row, 0 = w * 16) the call is asynchronous on `stream` for
        device memory and None is returned in place of the array."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        if row_count is None:
            row_count = (h - row_start + row_stride - 1) // row_stride
        if out_ptr is None:
            if out is None:
                out = np.empty((row_count, w, 4), np.float32)
            out_ptr = out.ctypes.data
        st = Stats() if want_stats else None
        _check(lib().rt_render_rows_f32(scene.handle, C.byref(camera) if camera is not None else None, w, h, spp,
                                        row_start, row_stride, row_count, out_ptr, pitch, stream,
                                        C.byref(st) if st is not None else None))
        return (out, st) if want_stats else out

    @staticmethod
    def render_preview(options, scene, step, camera=None, out_ptr=None, stream=None):
        """Undersampled preview (rt_render_preview): one traced pixel per step x step block, 1 sample per pixel."""
        w, h = options.width, options.height
        out = None
        if out_ptr is None:
            out = np.empty((h, w, 4), np.uint8)
            out_ptr = out.ctypes.data
        _check(lib().rt_render_preview(scene.handle, C.byref(camera) if camera is not None else None, w, h, step,
                                       out_ptr, w * h * 4, stream))
        return out

    @staticmethod
    def render_sweep(options, scene, n_frames, cameras=None, on_frame=None, rgb=False):
        """n_frames frames, copy of frame f overlapping the render of f+1; on_frame(f, array) per frame.
        rgb=True delivers (h, w, 3) frames packed on the device (the P6 file body)."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        cams = None
        if cameras is not None:
            cams = (Camera * n_frames)(*cameras)

        def _cb(user, frame, ptr, nbytes):
            if on_frame is not None:
                on_frame(int(frame), np.ctypeslib.as_array(ptr, shape=(h, w, 3 if rgb else 4)))

        cb = FRAME_CALLBACK(_cb)
        st = Stats()
        fn = lib().rt_render_sweep_rgb if rgb else lib().rt_render_sweep
        _check(fn(scene.handle, cams, n_frames, w, h, spp, cb, None, C.byref(st)))
        return st

    @staticmethod
    def render_sweep_pull(options, scene, next_frame, on_frame=None, rgb=False):
        """Sweep whose frames are pulled: next_frame() -> (frame_id, Camera or None = the reference camera), or
        None when nothing is left; on_frame(frame_id, array) per delivered frame (in pull order)."""
        w, h, spp = options.width, options.height, options.samples_per_pixel

        def _next(user, cam_out, use_cam):
            nxt = next_frame()
            if nxt is None:
                return -1
            if nxt[1] is None:
                use_cam[0] = 0
            else:
                C.memmove(cam_out, C.byref(nxt[1]), C.sizeof(Camera))
            return int(nxt[0])

        def _cb(user, frame, ptr, nbytes):
            if on_frame is not None:
                on_frame(int(frame), np.ctypeslib.as_array(ptr, shape=(h, w, 3 if rgb else 4)))

        nx, cb = NEXT_FRAME_CALLBACK(_next), FRAME_CALLBACK(_cb)
        st = Stats()
        _check(lib().rt_render_sweep_pull(scene.handle, nx, None, w, h, spp, 1 if rgb else 0, cb, None, C.byref(st)))
        return st

    @staticmethod
    def render_sweep_multi(options, scenes, n_frames, cameras=None, on_frame=None, rgb=False):
        """The sweep sharded by frame over len(scenes) GPUs of this process (the GPUs draw frames from one queue);
        on_frame(f, array) is called in frame order on the calling thread."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        cams = (Camera * n_frames)(*cameras) if cameras is not None else None

        def _cb(user, frame, ptr, nbytes):
            if on_frame is not None:
                on_frame(int(frame), np.ctypeslib.as_array(ptr, shape=(h, w, 3 if rgb else 4)))

        cb = FRAME_CALLBACK(_cb)
        st = Stats()
        arr = (C.c_void_p * len(scenes))(*[s.handle for s in scenes])
        _check(lib().rt_render_sweep_multi(arr, len(scenes), cams, n_frames, w, h, spp, 1 if rgb else 0, cb, None,
                                           C.byref(st)))
        return st

    @staticmethod
    def render_sweep_png(options, scenes, n_frames, cameras=None, on_frame=None):
        """The frame-sharded sweep (render_sweep_multi) delivering every frame as a PNG file encoded on its GPU:
        on_frame(f, bytes) in frame order on the calling thread; one scene is the single-GPU sweep."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        cams = (Camera * n_frames)(*cameras) if cameras is not None else None

        def _cb(user, frame, ptr, nbytes):
            if on_frame is not None:
                on_frame(int(frame), C.string_at(ptr, nbytes))

        cb = FRAME_CALLBACK(_cb)
        st = Stats()
        arr = (C.c_void_p * len(scenes))(*[s.handle for s in scenes])
        _check(lib().rt_render_sweep_png(arr, len(scenes), cams, n_frames, w, h, spp, cb, None, C.byref(st)))
        return st

    @staticmethod
    def render_sweep_apng(options, scenes, n_frames, cameras=None, fps=24, on_frame=None):
        """The frame-sharded sweep (render_sweep_multi) as one animated PNG showing `fps` frames a second:
        on_frame(f, bytes) receives frame f's payload in frame order on the calling thread, and the payloads joined
        in that order are the file.  One scene is the single-GPU sweep."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        cams = (Camera * n_frames)(*cameras) if cameras is not None else None

        def _cb(user, frame, ptr, nbytes):
            if on_frame is not None:
                on_frame(int(frame), C.string_at(ptr, nbytes))

        cb = FRAME_CALLBACK(_cb)
        st = Stats()
        arr = (C.c_void_p * len(scenes))(*[s.handle for s in scenes])
        _check(lib().rt_render_sweep_apng(arr, len(scenes), cams, n_frames, w, h, spp, 1, fps, cb, None, C.byref(st)))
        return st

    @staticmethod
    def render_multi(options, scenes, camera=None, want_stats=False):
        """Whole frame on len(scenes) GPUs of this process, rows interleaved, gathered on GPU 0."""
        w, h, spp = options.width, options.height, options.samples_per_pixel
        out = np.empty((h, w, 4), np.uint8)
        arr = (C.c_void_p * len(scenes))(*[s.handle for s in scenes])
        st = Stats() if want_stats else None
        _check(lib().rt_render_frame_multi(arr, len(scenes), C.byref(camera) if camera is not None else None, w, h,
                                           spp, out.ctypes.data, out.nbytes, C.byref(st) if st is not None else None))
        return (out, st) if want_stats else out


def measure_fp32_peak(device=0):
    t, c = C.c_double(), C.c_double()
    _check(lib().rt_measure_fp32_peak(device, C.byref(t), C.byref(c)))
    return t.value, c.value


def microbench_fp32(device, mode):
    t = C.c_double()
    _check(lib().rt_microbench_fp32(device, mode, C.byref(t)))
    return t.value


def microbench_d2h(nbytes, iters=24, n_buffers=3):
    """Copy-only device-to-host rate of the current device into a ring of pinned host buffers, GB/s."""
    g = C.c_double()
    _check(lib().rt_microbench_d2h(nbytes, iters, n_buffers, C.byref(g)))
    return g.value


def atomic_fetch_add_u64(addr, value=1):
    return int(lib().rt_atomic_fetch_add_u64(C.c_void_p(addr), value))


def host_register(ptr, nbytes):
    _check(lib().rt_host_register(C.c_void_p(ptr), nbytes))


def host_unregister(ptr):
    _check(lib().rt_host_unregister(C.c_void_p(ptr)))


def selftest_math(n=1 << 24, seed=1):
    m = (C.c_uint64 * 6)()
    _check(lib().rt_selftest_math(n, seed, m))
    return tuple(int(v) for v in m)


def debug_phased_tiles(scene):
    """(n_tiles, 2) uint32 array: primary / shadow candidates per cull tile of the last PHASED frame.
    0xffffffff marks a tile rendered by the per-lane walk, 0xfffffffd (shadow column) a tile whose shadow rays
    one leaf occludes (no list, no test).  n_tiles is the capacity of the tile-header buffer, which only grows:
    the last frame's tiles are the first rows."""
    n = C.c_uint32()
    L = lib()
    L.rt_debug_phased_tiles.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p]
    _check(L.rt_debug_phased_tiles(scene.handle, 0, C.byref(n), None))
    out = np.zeros((n.value, 2), dtype=np.uint32)
    _check(L.rt_debug_phased_tiles(scene.handle, n.value, C.byref(n), out.ctypes.data))
    return out


def device_alloc(nbytes):
    p = C.c_void_p()
    _check(lib().rt_device_alloc(nbytes, C.byref(p)))
    return p.value


def device_free(ptr):
    lib().rt_device_free(C.c_void_p(ptr))


def ipc_export(ptr):
    h = C.create_string_buffer(64)
    _check(lib().rt_ipc_export(C.c_void_p(ptr), h))
    return h.raw


def ipc_open(handle):
    p = C.c_void_p()
    _check(lib().rt_ipc_open(C.create_string_buffer(handle, 64), C.byref(p)))
    return p.value


def memcpy(dst, src, nbytes):
    _check(lib().rt_memcpy(C.c_void_p(dst), C.c_void_p(src), nbytes))


def pack_rgb_rows(rgba_ptr, rgb_ptr, width, height, row_start, row_stride, row_block, stream=None):
    _check(lib().rt_pack_rgb_rows(C.c_void_p(rgba_ptr), C.c_void_p(rgb_ptr), width, height, row_start, row_stride,
                                  row_block, stream))


def memcpy2d_async(dst, dpitch, src, spitch, width_bytes, rows, stream=None):
    _check(lib().rt_memcpy2d_async(C.c_void_p(dst), dpitch, C.c_void_p(src), spitch, width_bytes, rows, stream))


def png_bound(width, height):
    """Worst-case size of encode_png's file for a width x height frame (pure arithmetic, no device needed)."""
    n = C.c_size_t()
    _check(lib().rt_png_bound(width, height, C.byref(n)))
    return n.value


def encode_png(device_ptr, width, height, pitch=0, stream=None):
    """PNG file (bytes) of a width x height RGBA8 frame in device memory of the current device (alpha dropped),
    encoded on the GPU (rt_encode_png); waits for `stream`."""
    cap = png_bound(width, height)
    out = C.create_string_buffer(cap)
    n = C.c_size_t()
    _check(lib().rt_encode_png(C.c_void_p(device_ptr), width, height, pitch, out, cap, C.byref(n), stream))
    return out.raw[:n.value]


def apng_bound(width, height, n_frames):
    """Worst-case size of one frame's payload of encode_apng_frame (pure arithmetic, no device needed)."""
    n = C.c_size_t()
    _check(lib().rt_apng_bound(width, height, n_frames, C.byref(n)))
    return n.value


def encode_apng_frame(device_ptr, width, height, frame, n_frames, fps=24, pitch=0, stream=None):
    """Payload (bytes) of frame `frame` of an n_frames animated PNG showing `fps` frames a second, from a
    width x height RGBA8 frame in device memory of the current device, encoded on the GPU (rt_encode_apng_frame);
    the payloads of frames 0 .. n_frames-1 joined in order are the file.  Waits for `stream`."""
    cap = apng_bound(width, height, n_frames)
    out = C.create_string_buffer(cap)
    n = C.c_size_t()
    _check(lib().rt_encode_apng_frame(C.c_void_p(device_ptr), width, height, pitch, frame, n_frames, 1, fps, out, cap,
                                      C.byref(n), stream))
    return out.raw[:n.value]


def ipc_close(ptr):
    _check(lib().rt_ipc_close(C.c_void_p(ptr)))


class PinnedBuffer:
    """Pinned host memory from rt_host_alloc, exposed as a numpy array."""

    def __init__(self, nbytes):
        self._p = C.c_void_p()
        _check(lib().rt_host_alloc(nbytes, C.byref(self._p)))
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_uint8)), shape=(nbytes,))

    @property
    def ptr(self):
        return self._p.value

    def close(self):
        if self._p:
            self.array = None
            lib().rt_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
