"""The CPU oracle's AOV pixels (tests/_oracle_aov.cpp) over ctypes.  TEST INFRASTRUCTURE.

The library is the pinned oracle (oracle/oracle_rt.cpp, included unchanged) plus orc_render_rows_aov, compiled on
first use with oracle/Makefile's flags (the float oracle's, tests/_oracle_f32.py) into a directory under the system's
temporary directory, named after a hash of the sources and flags (the repository tree may be read-only).  Its scenes
are its own: Scene mirrors _oracle.Scene's constructors and adds render_aov.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import _oracle
import _oracle_f32

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "_oracle_aov.cpp"), os.path.join(_oracle.ORACLE_DIR, "oracle_rt.cpp"),
           os.path.join(_oracle.ORACLE_DIR, "oracle_rt.h")]
FLAGS = _oracle_f32.FLAGS

_lib = None


def build():
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for p in SOURCES:
        h.update(open(p, "rb").read())
    out_dir = os.path.join(tempfile.gettempdir(), "rtrace_oracle_aov_%s" % h.hexdigest()[:16])
    path = os.path.join(out_dir, "liboracle_aov.so")
    if not os.path.exists(path):
        os.makedirs(out_dir, exist_ok=True)
        tmp = "%s.%d" % (path, os.getpid())
        subprocess.check_call([os.environ.get("CXX", "g++")] + FLAGS + ["-I", _oracle.ORACLE_DIR, SOURCES[0], "-o", tmp])
        os.replace(tmp, path)   # atomic: a concurrent build never sees half a library
    return path


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build())
    vp, u32, f32p = C.c_void_p, C.c_uint32, C.POINTER(C.c_float)
    L.orc_scene_create.restype = vp
    L.orc_scene_create.argtypes = [u32, f32p, C.c_float, f32p, f32p]
    L.orc_scene_create_from_nodes.restype = vp
    L.orc_scene_create_from_nodes.argtypes = [u32, f32p, C.POINTER(u32), f32p, f32p]
    L.orc_scene_destroy.argtypes = [vp]
    L.orc_render_rows_aov.argtypes = [vp, C.POINTER(_oracle.Camera), u32, u32, u32, u32, u32, u32, u32, f32p]
    _lib = L
    return L


class Scene:
    """A scene of the AOV oracle; the constructors take _oracle.Scene's arguments."""

    def __init__(self, level=8, origin=(0.0, -1.0, 0.0), radius=1.0, light=(-1.0, -3.0, 2.0), eye=(0.0, 0.0, -4.0),
                 _handle=None):
        L = lib()
        self._h = _handle if _handle is not None else L.orc_scene_create(level, _oracle._f3(origin), radius,
                                                                         _oracle._f3(light), _oracle._f3(eye))
        if not self._h:
            raise ValueError("oracle scene creation failed (level must be > 1)")

    @classmethod
    def from_nodes(cls, spheres4, skip, light, eye):
        sph = np.ascontiguousarray(spheres4, dtype=np.float32)
        sk = np.ascontiguousarray(skip, dtype=np.uint32)
        h = lib().orc_scene_create_from_nodes(len(sk), _oracle._fp(sph), sk.ctypes.data_as(C.POINTER(C.c_uint32)),
                                              _oracle._f3(light), _oracle._f3(eye))
        return cls(_handle=h)

    def __del__(self):
        try:
            if self._h:
                lib().orc_scene_destroy(self._h)
        except Exception:
            pass
        self._h = None

    def render_aov(self, width, height, spp, row_start=0, row_stride=1, row_count=None, threads=None, camera=None):
        """The geometry of each pixel (include/rtrace.h "geometry output"): (row_count, width, 8) float32
        {nx, ny, nz, coverage, distance, px, py, pz}."""
        threads = threads or os.cpu_count() or 1
        if row_count is None:
            row_count = (height - row_start + row_stride - 1) // row_stride
        out = np.empty((row_count, width, 8), np.float32)
        lib().orc_render_rows_aov(self._h, C.byref(camera) if camera is not None else None, width, height, spp,
                                  row_start, row_stride, row_count, threads, _oracle._fp(out))
        return out
