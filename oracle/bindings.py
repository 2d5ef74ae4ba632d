"""ctypes bindings of the ORACLE -- test infrastructure, never imported by the product package.

Only tests/, __graft_entry__.smoke() and bench.py's reference / cpu_baseline legs import this module.

* ``Reference``   -> oracle/_ref/libraylib_ref.so (+ oracle/_ref/libscenes_ref.so): the unmodified reference sources
  compiled where they lie (oracle/Makefile) with the deterministic RNG shim, bound through the SAME reference C ABI
  as the product (raylib/raylib.h:23-149) plus the oracle driver's entry points (oracle/oracle_driver.cc).
* ``Restatement`` -> oracle/lib/librt_oracle.so: the plain-C restatement of closest hit + camera rays on the
  flattened scene (oracle/rt_oracle.c).
"""
import ctypes as C
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "software-raytracing_b200"))
from pyraylib import (_Base, _bind, _F32P, _I32P, H, RendererSettings, RtCamera, RtSceneDesc)  # noqa: E402

REF_LIB = os.path.join(HERE, "_ref", "libraylib_ref.so")
REF_SCENES = os.path.join(HERE, "_ref", "libscenes_ref.so")
RESTATE_LIB = os.path.join(HERE, "lib", "librt_oracle.so")
# scenes/scenes.cc compiled against the REFERENCE's headers, linked against the product library (oracle/Makefile)
XABI_SCENES = os.path.join(HERE, "_ref", "libscenes_xabi.so")


class OracleRenderStats(C.Structure):
    _fields_ = [("rayQueries", C.c_uint64), ("rngDraws", C.c_uint64), ("seconds", C.c_double),
                ("threads", C.c_int32), ("debugbreaks", C.c_int32)]


class OraclePrimaryStats(C.Structure):
    _fields_ = [("boxTests", C.c_uint64), ("triTests", C.c_uint64), ("sphereTests", C.c_uint64),
                ("otherTests", C.c_uint64), ("rays", C.c_uint64), ("walkVsHitMismatches", C.c_uint64),
                ("numLeaves", C.c_int32), ("maxDepth", C.c_int32), ("numNodes", C.c_int32), ("pad", C.c_int32),
                ("seconds", C.c_double)]



ORACLE_API = {
    "oracle_rng_reset": (None, [C.c_uint64]),
    "oracle_hardware_threads": (C.c_int32, []),
    "oracle_render": (None, [C.POINTER(RendererSettings), H, H, H, C.c_uint64, C.c_int32, C.POINTER(OracleRenderStats)]),
    "oracle_render_region": (None, [C.POINTER(RendererSettings), H, H, H, C.c_uint64, C.c_int32,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(OracleRenderStats)]),
    "oracle_native_render": (C.c_double, [C.POINTER(RendererSettings), H, H, H, C.POINTER(OracleRenderStats)]),
    "oracle_primary_hits": (None, [C.POINTER(RendererSettings), H, H, C.c_uint64, C.c_int32, _I32P, _F32P, C.c_void_p,
                                   C.POINTER(OraclePrimaryStats)]),
    "oracle_trace_rays": (None, [H, _F32P, C.c_int64, C.c_float, C.c_int32, _I32P, _F32P, C.POINTER(OraclePrimaryStats)]),
    "oracle_forget_scene": (None, [H]),
    "oracle_debugbreak_count": (C.c_long, []),
    "oracle_image_set_rgba": (None, [H, C.c_uint32, C.c_uint32, _F32P]),
    "oracle_image_get_rgba": (None, [H, _F32P]),
}



class Reference(_Base):
    """The compiled reference + deterministic driver (oracle/_ref). Test infrastructure."""

    def __init__(self):
        super().__init__(REF_LIB, REF_SCENES)
        _bind(self.lib, ORACLE_API)

    def render_deterministic(self, settings, scene, camera, seed=1337, threads=0, region=None):
        img = self.lib.Raylib_CreateImage(settings.viewportWidth, settings.viewportHeight)
        st = OracleRenderStats()
        try:
            if region is None:
                self.lib.oracle_render(C.byref(settings), scene, camera, img, seed, threads, C.byref(st))
            else:
                x0, y0, x1, y1 = region
                self.lib.oracle_render_region(C.byref(settings), scene, camera, img, seed, threads, x0, y0, x1, y1, C.byref(st))
            return self.dump_image(img, settings.viewportWidth, settings.viewportHeight), st
        finally:
            self.lib.Raylib_DestroyImage(img)

    def postprocess_rgba(self, rgba):
        """The reference's own Raylib_PostProcess (Image2D::PostProcess, render/image.cc:44-103) on an H x W x 4 frame."""
        rgba = np.ascontiguousarray(rgba, dtype=np.float32)
        h, w = rgba.shape[:2]
        img = self.lib.Raylib_CreateImage(w, h)
        try:
            self.lib.oracle_image_set_rgba(img, w, h, rgba)
            self.lib.Raylib_PostProcess(img)
            out = np.empty_like(rgba)
            self.lib.oracle_image_get_rgba(img, out)
            return out
        finally:
            self.lib.Raylib_DestroyImage(img)

    def render_native(self, settings, scene, camera):
        """The reference's own Renderer::RenderScene (thread pool, non-deterministic work split)."""
        img = self.lib.Raylib_CreateImage(settings.viewportWidth, settings.viewportHeight)
        st = OracleRenderStats()
        try:
            sec = self.lib.oracle_native_render(C.byref(settings), scene, camera, img, C.byref(st))
            return self.dump_image(img, settings.viewportWidth, settings.viewportHeight), sec
        finally:
            self.lib.Raylib_DestroyImage(img)

    def primary_hits(self, settings, scene, camera, seed=1337, threads=0, want_rays=False):
        n = settings.viewportWidth * settings.viewportHeight
        rank = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        rays = np.empty((n, 8), dtype=np.float32) if want_rays else None
        st = OraclePrimaryStats()
        self.lib.oracle_primary_hits(C.byref(settings), scene, camera, seed, threads, rank, t,
                                     rays.ctypes.data if want_rays else None, C.byref(st))
        return rank, t, rays, st

    def trace_rays(self, scene, rays, t_min, threads=0):
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 8)
        rank = np.empty(len(rays), dtype=np.int32)
        t = np.empty(len(rays), dtype=np.float32)
        st = OraclePrimaryStats()
        self.lib.oracle_trace_rays(scene, rays, len(rays), t_min, threads, rank, t, C.byref(st))
        return rank, t, st


class Restatement:
    """oracle/rt_oracle.c: plain-C closest hit + camera rays on the flattened scene. Test infrastructure."""

    def __init__(self):
        if not os.path.exists(RESTATE_LIB):
            raise RuntimeError("%s is missing -- run __graft_entry__.build()" % RESTATE_LIB)
        self.lib = C.CDLL(RESTATE_LIB)
        self.lib.rt_oracle_trace.restype = None
        self.lib.rt_oracle_trace.argtypes = [C.POINTER(RtSceneDesc), _F32P, C.c_int64, C.c_float, _I32P, _F32P,
                                             C.POINTER(C.c_uint64 * 4)]
        self.lib.rt_oracle_primary.restype = None
        self.lib.rt_oracle_primary.argtypes = [C.POINTER(RtSceneDesc), C.POINTER(RtCamera), C.c_uint32, C.c_uint32,
                                               C.c_uint32, C.c_uint32, C.c_float, C.c_uint64, _I32P, _F32P, C.c_void_p,
                                               C.POINTER(C.c_uint64 * 4)]

    def check_quantization(self, desc):
        self.lib.rt_oracle_check_quantization.restype = C.c_uint64
        self.lib.rt_oracle_check_quantization.argtypes = [C.POINTER(RtSceneDesc)]
        return int(self.lib.rt_oracle_check_quantization(desc))

    def select_tree(self, which):
        """0/False: reference topology (default). 1/True: the binary SAH tree, visited exhaustively.
        2: that tree collapsed to 4-wide nodes (exact boxes).  3: the quantized 64-byte nodes the device walks, decoded to
        boxes.  4: the same nodes with the device's own conservative ray-space test (rt_traverse.cuh trav_step)."""
        self.lib.rt_oracle_select_tree(int(which))

    def trace(self, desc, rays, t_min):
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 8)
        rank = np.empty(len(rays), dtype=np.int32)
        t = np.empty(len(rays), dtype=np.float32)
        counts = (C.c_uint64 * 4)()
        self.lib.rt_oracle_trace(desc, rays, len(rays), t_min, rank, t, C.byref(counts))
        return rank, t, list(counts)

    def trace_hits(self, desc, rays, t_min):
        """trace() plus what a device hit record and queue hold: -> (rank, t, uv n x 2 (paramU / paramV of triangle hits,
        else 0), face (0..5 of cube hits in the device's order, else -1), material type of the hit primitive (-1: miss),
        counts)."""
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 8)
        n = len(rays)
        rank = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        uv = np.empty((n, 2), dtype=np.float32)
        face = np.empty(n, dtype=np.int32)
        mat = np.empty(n, dtype=np.int32)
        counts = (C.c_uint64 * 4)()
        fn = self.lib.rt_oracle_trace_hits
        fn.restype = None
        fn.argtypes = [C.POINTER(RtSceneDesc), _F32P, C.c_int64, C.c_float, _I32P, _F32P, _F32P, _I32P, _I32P,
                       C.POINTER(C.c_uint64 * 4)]
        fn(desc, rays, n, t_min, rank, t, uv, face, mat, C.byref(counts))
        return rank, t, uv, face, mat, list(counts)

    def primary(self, desc, cam, width, height, t_min, seed=1337, rows=None, want_rays=False):
        """want_rays: also return the n x 8 camera rays (bit-identical to the compiled reference's, tests/golden)."""
        n = width * height
        rank = np.full(n, -2, dtype=np.int32)
        t = np.zeros(n, dtype=np.float32)
        rays = np.zeros((n, 8), dtype=np.float32) if want_rays else None
        counts = (C.c_uint64 * 4)()
        y0, y1 = rows if rows else (0, height)
        self.lib.rt_oracle_primary(desc, C.byref(cam), width, height, y0, y1, t_min, seed, rank, t,
                                   rays.ctypes.data if want_rays else None, C.byref(counts))
        return (rank, t, list(counts), rays) if want_rays else (rank, t, list(counts))
