"""ctypes bindings of the product library, used by tests/, bench.py and __graft_entry__.py.

``Product`` -> software-raytracing_b200/lib/libraylib_b200.so (+ scenes/lib/libscenes_b200.so), bound through the
reference C ABI (raylib/raylib.h:23-149) plus the RaylibB200_* additions (include/raylib_b200.h).

The product never falls back to anything: if the CUDA library is missing or no device is visible, render calls
raise.  The bindings of the oracle (compiled reference, C restatement) live in oracle/bindings.py -- test
infrastructure that this module never imports.
"""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

PRODUCT_LIB = os.path.join(HERE, "lib", "libraylib_b200.so")
PRODUCT_SCENES = os.path.join(ROOT, "scenes", "lib", "libscenes_b200.so")

RENDERMODE = {"Default": 0, "Albedo": 1, "SurfaceNormal": 2, "MicrosurfaceNormal": 3, "Texcoord": 4,
              "Emission": 5, "Reflectance": 6}


class RendererSettings(C.Structure):
    _fields_ = [("viewportWidth", C.c_uint32), ("viewportHeight", C.c_uint32),
                ("samplesPerPixel", C.c_int32), ("maxPathLength", C.c_int32),
                ("rayTMin", C.c_float), ("renderMode", C.c_uint32)]

    def copy(self, **kw):
        s = RendererSettings(self.viewportWidth, self.viewportHeight, self.samplesPerPixel,
                             self.maxPathLength, self.rayTMin, self.renderMode)
        for k, v in kw.items():
            setattr(s, k, v)
        return s


class DemoSceneInfo(C.Structure):
    _fields_ = [("scene", C.c_size_t), ("camera", C.c_size_t), ("settings", RendererSettings),
                ("numTriangles", C.c_uint64), ("numSpheres", C.c_uint64), ("numMeshes", C.c_uint64),
                ("cameraPos", C.c_float * 3), ("cameraLookAt", C.c_float * 3),
                ("fovY", C.c_float), ("aperture", C.c_float), ("focalDistance", C.c_float),
                ("shutterBegin", C.c_float), ("shutterEnd", C.c_float)]


class B200Stats(C.Structure):
    _fields_ = [("rayQueries", C.c_uint64), ("pixelSamples", C.c_uint64),
                ("boxTests", C.c_uint64), ("triTests", C.c_uint64), ("sphereTests", C.c_uint64), ("nodeVisits", C.c_uint64),
                ("refBoxTests", C.c_uint64), ("refTriTests", C.c_uint64), ("refSphereTests", C.c_uint64), ("statRays", C.c_uint64),
                ("deviceMs", C.c_double), ("extendMs", C.c_double), ("extendLaunches", C.c_uint32), ("pad0", C.c_uint32),
                ("totalMs", C.c_double),
                ("h2dBytes", C.c_uint64), ("d2hBytes", C.c_uint64),
                ("kernelLaunches", C.c_uint32), ("passes", C.c_uint32), ("device", C.c_uint32), ("devicesUsed", C.c_uint32),
                ("nodeIters", C.c_uint64), ("nodeStep", C.c_uint64), ("nodeAlive", C.c_uint64), ("leafIters", C.c_uint64), ("leafBusy", C.c_uint64),
                ("gateTests", C.c_uint64), ("cubeTests", C.c_uint64)]


class RtCamera(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("lensRadius", C.c_float),
                ("topLeft", C.c_float * 3), ("beginTime", C.c_float),
                ("horizontal", C.c_float * 3), ("timePeriod", C.c_float),
                ("vertical", C.c_float * 3), ("pad0", C.c_float),
                ("u", C.c_float * 3), ("pad1", C.c_float),
                ("v", C.c_float * 3), ("pad2", C.c_float)]


class RtSceneDesc(C.Structure):
    _fields_ = [("nodes", C.c_void_p), ("numNodes", C.c_uint32),
                ("triHot", C.c_void_p), ("triCold", C.c_void_p), ("triRank", C.c_void_p), ("numTris", C.c_uint32),
                ("triGate", C.c_void_p), ("gateBoxes", C.c_void_p), ("numGates", C.c_uint32),
                ("sphereGate", C.c_void_p), ("cubeGate", C.c_void_p),
                ("spheres", C.c_void_p), ("sphereMaterial", C.c_void_p), ("sphereRank", C.c_void_p), ("numSpheres", C.c_uint32),
                ("cubes", C.c_void_p), ("cubeRank", C.c_void_p), ("numCubes", C.c_uint32),
                ("materials", C.c_void_p), ("numMaterials", C.c_uint32),
                ("textures", C.c_void_p), ("numTextures", C.c_uint32),
                ("texels", C.c_void_p), ("numTexels", C.c_uint64),
                ("rootMin", C.c_float * 3), ("rootMax", C.c_float * 3),
                ("rootRef", C.c_uint32), ("maxStackDepth", C.c_uint32), ("treeKind", C.c_uint32),
                ("wideNodes", C.c_void_p), ("numWideNodes", C.c_uint32), ("quantNodes", C.c_void_p), ("wideRootRef", C.c_uint32), ("wideMaxStack", C.c_uint32),
                ("refNodes", C.c_void_p), ("numRefNodes", C.c_uint32),
                ("refRootMin", C.c_float * 3), ("refRootMax", C.c_float * 3),
                ("refRootRef", C.c_uint32), ("refRootBoxTests", C.c_uint32), ("refMaxDepth", C.c_uint32),
                ("flags", C.c_uint32),
                ("materialTypeMask", C.c_uint32), ("numLeaves", C.c_uint32),
                ("skyTexture", C.c_int32), ("skyRotation", C.c_float * 9),
                ("sunIlluminance", C.c_float * 3), ("sunDirection", C.c_float * 3)]


# Product and reference export the same symbol names; keep each library in its own lookup scope.
_DLMODE = os.RTLD_LOCAL | os.RTLD_NOW | getattr(os, "RTLD_DEEPBIND", 0)

H = C.c_size_t      # uintptr_t handles
_F32P = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_I32P = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")

# The reference C ABI: name -> (restype, argtypes).  raylib/raylib.h:23-149
RAYLIB_C_API = {
    "Raylib_Initialize": (C.c_int32, []),
    "Raylib_Terminate": (C.c_int32, []),
    "Raylib_LoadOBJModel": (H, [C.c_char_p]),
    "Raylib_TransformOBJModel": (None, [H] + [C.c_float] * 9),
    "Raylib_FinalizeOBJModel": (None, [H]),
    "Raylib_UnloadOBJModel": (C.c_int32, [H]),
    "Raylib_LoadImage": (H, [C.c_char_p]),
    "Raylib_CreateScene": (H, []),
    "Raylib_AddSceneElement": (None, [H, H]),
    "Raylib_AddOBJModelToScene": (None, [H, H]),
    "Raylib_SetSkyPanorama": (None, [H, H]),
    "Raylib_SetSunIlluminance": (None, [H, C.c_float, C.c_float, C.c_float]),
    "Raylib_SetSunDirection": (None, [H, C.c_float, C.c_float, C.c_float]),
    "Raylib_FinalizeScene": (None, [H]),
    "Raylib_DestroyScene": (C.c_int32, [H]),
    "Raylib_CreateCamera": (H, []),
    "Raylib_CameraSetPosition": (None, [H, C.c_float, C.c_float, C.c_float]),
    "Raylib_CameraSetLookAt": (None, [H, C.c_float, C.c_float, C.c_float]),
    "Raylib_CameraSetPerspective": (None, [H, C.c_float, C.c_float]),
    "Raylib_CameraSetLens": (None, [H, C.c_float, C.c_float]),
    "Raylib_CameraSetMotion": (None, [H, C.c_float, C.c_float]),
    "Raylib_CameraCopy": (None, [H, H]),
    "Raylib_DestroyCamera": (C.c_int32, [H]),
    "Raylib_CreateImage": (H, [C.c_uint32, C.c_uint32]),
    "Raylib_DumpImageData": (None, [H, _F32P]),
    "Raylib_DestroyImage": (C.c_int32, [H]),
    "Raylib_Render": (None, [C.POINTER(RendererSettings), H, H, H]),
    "Raylib_Denoise": (C.c_int32, [H, C.c_int32, H, H, H]),
    "Raylib_PostProcess": (None, [H]),
    "Raylib_IsDenoiserSupported": (C.c_int32, []),
    "Raylib_GetRenderModeString": (C.c_char_p, [C.c_uint32]),
    "Raylib_WriteImageToDisk": (C.c_int32, [H, C.c_char_p, C.c_uint32]),
    "Raylib_FlushLogThread": (None, []),
}

B200_C_API = {
    "RaylibB200_DeviceCount": (C.c_int32, []),
    "RaylibB200_SetDevice": (C.c_int32, [C.c_int32]),
    "RaylibB200_GetDevice": (C.c_int32, []),
    "RaylibB200_SetDevices": (C.c_int32, [C.c_int32]),
    "RaylibB200_GetDeviceCountInUse": (C.c_int32, []),
    "RaylibB200_ReloadTuning": (None, []),
    "RaylibB200_SetFrameSeed": (None, [C.c_uint64]),
    "RaylibB200_SetBvhBuildKey": (None, [C.c_uint64]),
    "RaylibB200_SetCollectStats": (None, [C.c_int32]),
    "RaylibB200_SetTimeStages": (None, [C.c_int32]),
    "RaylibB200_SetSamplesPerPass": (None, [C.c_uint32]),
    "RaylibB200_SetPipes": (None, [C.c_uint32]),
    "RaylibB200_SetFusedPass": (None, [C.c_uint32]),
    "RaylibB200_GetLastStats": (C.c_int32, [C.POINTER(B200Stats)]),
    "RaylibB200_GetLastError": (C.c_char_p, []),
    "RaylibB200_SceneDeviceBytes": (C.c_uint64, [H]),
    "RaylibB200_SceneCounts": (C.c_int32, [H, C.POINTER(C.c_uint64 * 8)]),
    "RaylibB200_ShardPixelCapacity": (C.c_uint64, [C.c_uint32, C.c_uint32, C.c_uint32]),
    "RaylibB200_RenderShard": (C.c_int32, [C.POINTER(RendererSettings), H, H, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "RaylibB200_AssembleShards": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "RaylibB200_RenderShardToFrame": (C.c_int32, [C.POINTER(RendererSettings), H, H, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "RaylibB200_FrameCreate": (C.c_void_p, [C.c_uint32, C.c_uint32, C.c_void_p]),
    "RaylibB200_FrameDestroy": (None, [C.c_void_p]),
    "RaylibB200_FrameOpen": (C.c_void_p, [C.c_void_p]),
    "RaylibB200_FrameClose": (C.c_int32, [C.c_void_p]),
    "RaylibB200_FrameRead": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "RaylibB200_ShardPixelMap": (C.c_int32, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")]),
    "RaylibB200_AssembleShardsHost": (C.c_int32, [_F32P, C.c_uint32, C.c_uint32, C.c_uint32, _F32P]),
    "RaylibB200_RenderToDevice": (C.c_int32, [C.POINTER(RendererSettings), H, H, C.c_void_p, C.c_void_p]),
    "RaylibB200_RenderAux": (C.c_int32, [C.POINTER(RendererSettings), H, H, H, H]),
    "RaylibB200_PostProcessDevice": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_float), C.c_void_p]),
    "RaylibB200_PostProcessGPU": (C.c_int32, [H]),
    "RaylibB200_LibmEval": (C.c_int32, [C.c_int32, _F32P, C.c_void_p, _F32P, C.c_uint64]),
    "RaylibB200_ImageSetRGBA": (C.c_int32, [H, C.c_uint32, C.c_uint32, _F32P]),
    "RaylibB200_ImageGetRGBA": (C.c_int32, [H, _F32P]),
    "RaylibB200_TraceRays": (C.c_int32, [H, _F32P, C.c_int64, C.c_float, _I32P, _F32P]),
    "RaylibB200_PrimaryHits": (C.c_int32, [C.POINTER(RendererSettings), H, H, _I32P, _F32P]),
    "RaylibB200_SaveFlattenedScene": (C.c_int32, [H, C.c_char_p]),
    "RaylibB200_LoadFlattenedScene": (H, [C.c_char_p]),
    "RaylibB200_FlattenForInspection": (C.POINTER(RtSceneDesc), [H]),
    "RaylibB200_ReleaseInspection": (None, [H]),
    "RaylibB200_CameraBlock": (C.c_int32, [H, C.POINTER(RtCamera)]),
    "RaylibB200_SeedHostRandom": (None, [C.c_uint64]),
    "RaylibB200_AccumulatorCreate": (C.c_void_p, [C.c_uint32, C.c_uint32]),
    "RaylibB200_AccumulatorDestroy": (None, [C.c_void_p]),
    "RaylibB200_AccumulatorReset": (C.c_int32, [C.c_void_p]),
    "RaylibB200_AccumulatorSamples": (C.c_uint32, [C.c_void_p]),
    "RaylibB200_RenderAccumulate": (C.c_int32, [C.POINTER(RendererSettings), H, H, C.c_void_p, C.c_uint32]),
    "RaylibB200_AccumulatorResolve": (C.c_int32, [C.c_void_p, H]),
    "RaylibB200_AccumulatorResolveDevice": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "RaylibB200_AccumulatorRead": (C.c_int32, [C.c_void_p, _F32P]),
    "RaylibB200_AccumulatorNoise": (C.c_int32, [C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]),
    "RaylibB200_AccumulatorSave": (C.c_int32, [C.c_void_p, C.c_char_p]),
    "RaylibB200_AccumulatorLoad": (C.c_void_p, [C.c_char_p]),
    "RaylibB200_Denoise": (C.c_int32, [H, H, H, H]),
    "RaylibB200_DenoiseDevice": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "RaylibB200_AccumulatorDenoise": (C.c_int32, [C.c_void_p, H, H, H]),
}

SCENES_API = {
    "demo_scene_create": (C.c_int32, [C.c_int32, C.c_int32, C.POINTER(DemoSceneInfo)]),
    "demo_scene_destroy": (None, [H, H]),
    "demo_camera_set_aspect": (None, [H, C.c_float, C.c_uint32, C.c_uint32]),
}

def _bind(lib, table):
    for name, (res, args) in table.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args


class _Base:
    """Common scene/camera/image plumbing over the reference C ABI."""

    def __init__(self, lib_path, scenes_path):
        if not os.path.exists(lib_path):
            raise RuntimeError("%s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'`" % lib_path)
        self.lib = C.CDLL(lib_path, mode=_DLMODE)
        _bind(self.lib, RAYLIB_C_API)
        self.scenes = C.CDLL(scenes_path, mode=_DLMODE)
        _bind(self.scenes, SCENES_API)

    def create_demo(self, config, size_param=0):
        info = DemoSceneInfo()
        if not self.scenes.demo_scene_create(config, size_param, C.byref(info)):
            raise RuntimeError("demo_scene_create(%d) failed" % config)
        return info

    def destroy_demo(self, info):
        self.scenes.demo_scene_destroy(info.scene, info.camera)

    def set_viewport(self, info, width, height):
        """Render a configuration at another resolution (camera aspect follows)."""
        info.settings.viewportWidth = width
        info.settings.viewportHeight = height
        self.scenes.demo_camera_set_aspect(info.camera, info.fovY, width, height)

    def dump_image(self, image, width, height):
        out = np.empty((height, width, 3), dtype=np.float32)
        self.lib.Raylib_DumpImageData(image, out)
        return out

    def render(self, settings, scene, camera):
        """Raylib_Render through the reference C ABI; returns H x W x 3 float32."""
        img = self.lib.Raylib_CreateImage(settings.viewportWidth, settings.viewportHeight)
        try:
            self.lib.Raylib_Render(C.byref(settings), scene, camera, img)
            return self.dump_image(img, settings.viewportWidth, settings.viewportHeight)
        finally:
            self.lib.Raylib_DestroyImage(img)


class Product(_Base):
    def __init__(self, scenes_path=None):
        """scenes_path: another build of the scene client library bound to the same product library (tests load the
        cross-ABI client compiled against the reference's headers, oracle/_ref/libscenes_xabi.so)."""
        super().__init__(PRODUCT_LIB, scenes_path or PRODUCT_SCENES)
        _bind(self.lib, B200_C_API)

    def device_count(self):
        return int(self.lib.RaylibB200_DeviceCount())

    def require_gpu(self):
        if self.device_count() <= 0:
            raise RuntimeError("no CUDA device visible: libraylib_b200 renders on the GPU only")

    def last_error(self):
        return self.lib.RaylibB200_GetLastError().decode()

    def last_stats(self):
        st = B200Stats()
        if not self.lib.RaylibB200_GetLastStats(C.byref(st)):
            raise RuntimeError("no render statistics available: " + self.last_error())
        return st

    def render(self, settings, scene, camera):
        self.require_gpu()
        img = super().render(settings, scene, camera)
        err = self.last_error()
        if err:
            raise RuntimeError("Raylib_Render failed: " + err)
        return img

    def primary_hits(self, settings, scene, camera):
        self.require_gpu()
        n = settings.viewportWidth * settings.viewportHeight
        rank = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        if not self.lib.RaylibB200_PrimaryHits(C.byref(settings), scene, camera, rank, t):
            raise RuntimeError("RaylibB200_PrimaryHits failed: " + self.last_error())
        return rank, t

    def trace_rays(self, scene, rays, t_min):
        self.require_gpu()
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 8)
        rank = np.empty(len(rays), dtype=np.int32)
        t = np.empty(len(rays), dtype=np.float32)
        if not self.lib.RaylibB200_TraceRays(scene, rays, len(rays), t_min, rank, t):
            raise RuntimeError("RaylibB200_TraceRays failed: " + self.last_error())
        return rank, t

    def flat_desc(self, scene):
        p = self.lib.RaylibB200_FlattenForInspection(scene)
        if not p:
            raise RuntimeError("flatten failed: " + self.last_error())
        return p

    def camera_block(self, camera):
        cam = RtCamera()
        self.lib.RaylibB200_CameraBlock(camera, C.byref(cam))
        return cam

    # ---- progressive rendering (RaylibB200_Accumulator*): acc is the handle of RaylibB200_AccumulatorCreate / _Load
    def accumulate(self, settings, scene, camera, acc, samples):
        """Renders `samples` more samples of every pixel into the accumulator; raises when the call is refused."""
        if not self.lib.RaylibB200_RenderAccumulate(C.byref(settings), scene, camera, acc, samples):
            raise RuntimeError("RaylibB200_RenderAccumulate failed: " + self.last_error())

    def resolve(self, acc, width, height):
        """The running average (RaylibB200_AccumulatorResolve): H x W x 3 float32, the bits Raylib_Render gives at n spp."""
        img = self.lib.Raylib_CreateImage(1, 1)          # resized by the resolve, as Raylib_Render resizes its output
        try:
            if not self.lib.RaylibB200_AccumulatorResolve(acc, img):
                raise RuntimeError("RaylibB200_AccumulatorResolve failed: " + self.last_error())
            return self.dump_image(img, width, height)
        finally:
            self.lib.Raylib_DestroyImage(img)

    def accumulator_sums(self, acc, width, height):
        """Raw sums: H x W x 4 float32 {sum R, sum G, sum B, sum luminance^2}."""
        out = np.empty((height, width, 4), dtype=np.float32)
        if not self.lib.RaylibB200_AccumulatorRead(acc, out):
            raise RuntimeError("RaylibB200_AccumulatorRead failed: " + self.last_error())
        return out

    def noise(self, acc, width, height):
        """(H x W float32 relative standard error of each pixel's mean luminance, their mean as a float)."""
        out = np.empty((height, width), dtype=np.float32)
        mean = C.c_double()
        if not self.lib.RaylibB200_AccumulatorNoise(acc, out.ctypes.data, C.byref(mean)):
            raise RuntimeError("RaylibB200_AccumulatorNoise failed: " + self.last_error())
        return out, mean.value

    # ---- denoising (RaylibB200_Denoise, _DenoiseDevice, _AccumulatorDenoise): guides are the albedo and encoded-normal
    # views of RaylibB200_RenderAux, or None
    def image_from_array(self, a):
        """A new image handle holding an H x W x 3 or 4 float32 array (alpha 1 when absent); destroy with Raylib_DestroyImage."""
        a = np.asarray(a, dtype=np.float32)
        rgba = np.ones(a.shape[:2] + (4,), dtype=np.float32)
        rgba[:, :, :a.shape[2]] = a
        img = self.lib.Raylib_CreateImage(1, 1)
        self.lib.RaylibB200_ImageSetRGBA(img, a.shape[1], a.shape[0], rgba)
        return img

    def _denoise_host(self, call, name, height, width, guides):
        handles = [self.image_from_array(g) if g is not None else 0 for g in guides]
        out = self.lib.Raylib_CreateImage(1, 1)          # resized by the call
        try:
            if not call(*handles, out):
                raise RuntimeError(name + " failed: " + self.last_error())
            rgba = np.empty((height, width, 4), dtype=np.float32)
            self.lib.RaylibB200_ImageGetRGBA(out, rgba)
            return rgba[:, :, :3].copy()
        finally:
            for h in handles + [out]:
                if h:
                    self.lib.Raylib_DestroyImage(h)

    def denoise(self, color, albedo=None, normal=None):
        """RaylibB200_Denoise on H x W x 3 or 4 float32 arrays: H x W x 3 float32."""
        color = np.asarray(color, dtype=np.float32)
        main = self.image_from_array(color)
        try:
            return self._denoise_host(lambda a, n, out: self.lib.RaylibB200_Denoise(main, a, n, out), "RaylibB200_Denoise",
                                      color.shape[0], color.shape[1], (albedo, normal))
        finally:
            self.lib.Raylib_DestroyImage(main)

    def denoise_device(self, color, albedo=None, normal=None):
        """RaylibB200_DenoiseDevice on H x W x 4 float32 CUDA tensors (torch) of the current device, on torch's current
        stream: H x W x 3 float32 (numpy)."""
        import torch
        out = torch.empty_like(color)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        if not self.lib.RaylibB200_DenoiseDevice(ptr(color), ptr(albedo), ptr(normal), color.shape[1], color.shape[0], ptr(out),
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)):
            raise RuntimeError("RaylibB200_DenoiseDevice failed: " + self.last_error())
        return out[:, :, :3].cpu().numpy()

    def accumulator_denoise(self, acc, width, height, albedo=None, normal=None):
        """RaylibB200_AccumulatorDenoise with H x W x 3 or 4 float32 guide arrays: H x W x 3 float32."""
        return self._denoise_host(lambda a, n, out: self.lib.RaylibB200_AccumulatorDenoise(acc, a, n, out),
                                  "RaylibB200_AccumulatorDenoise", height, width, (albedo, normal))


def device_source_hash():
    """sha256 (first 16 hex digits) over the sources that decide what k_extend executes and walks: the device code, the
    scene format and the host tree pipeline.  profiles/traffic.json records it so that bench.py can refuse DRAM-traffic
    figures captured on another build."""
    import hashlib
    files = []
    for sub in ("csrc/device", "csrc/host"):
        d = os.path.join(HERE, sub)
        files += [os.path.join(d, f) for f in sorted(os.listdir(d))
                  if f.endswith((".cu", ".cuh")) or f in ("flatten.cc", "bvh_sah.cc", "bvh_sah.h")]
    files += [os.path.join(ROOT, "include", f) for f in ("rt_scene_format.h", "rt_device_abi.h", "rt_rng.h")]
    h = hashlib.sha256()
    for f in files:
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def psnr(a, b, peak=1.0):
    a = np.clip(np.nan_to_num(a.astype(np.float64)), 0.0, peak)
    b = np.clip(np.nan_to_num(b.astype(np.float64)), 0.0, peak)
    mse = float(np.mean((a - b) ** 2))
    return 99.0 if mse == 0.0 else 10.0 * np.log10(peak * peak / mse)
